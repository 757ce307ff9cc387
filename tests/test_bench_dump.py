"""bench.py --dump-outputs on the CPU: what dump_outputs writes for a batch of frames, and that it stays within 64 MB
at the benchmark's own 4096x3000 frame size."""
import numpy as np
import torch

import bench


def test_dump_outputs_last_frame_and_seeded_sample(tmp_path):
    out = torch.rand((3, 30, 41), generator=torch.Generator().manual_seed(5))
    bench.dump_outputs(str(tmp_path / 'a'), out)
    bench.dump_outputs(str(tmp_path / 'b'), out)
    last = np.load(tmp_path / 'a' / 'out_last_frame.npy')
    sample = np.load(tmp_path / 'a' / 'out_sample.npy')
    assert last.dtype == np.float32 and np.array_equal(last, out[-1].numpy())
    assert sample.dtype == np.float32 and sample.shape == (bench.DUMP_SAMPLE,)
    assert np.isin(sample, out.numpy()).all()
    for name in ('out_last_frame.npy', 'out_sample.npy'):
        assert np.array_equal(np.load(tmp_path / 'a' / name), np.load(tmp_path / 'b' / name))


def test_dump_outputs_fit_64_mb_at_the_benchmark_frame_size():
    assert (bench.H * bench.W + bench.DUMP_SAMPLE) * 4 + 2 * 128 <= 64e6
