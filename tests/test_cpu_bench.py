"""bench.py host logic: --steps is the number of timed steps, and --dump-outputs writes the same float32
arrays on every run with the same arguments (checked on the CPU arm, --impl reference)."""
import os
import subprocess
import sys

import numpy as np

import parity


def test_repeat_sizes_cover_exactly_the_timed_steps():
    import bench
    for k in (1, 7, 19, 20, 39, 40, 200, 301, 3000, 10 ** 5):
        sizes = bench.repeat_sizes(k, 15)
        assert sum(sizes) == k and 1 <= len(sizes) <= 15 and max(sizes) - min(sizes) <= 1
        assert len(sizes) == 1 or min(sizes) >= bench.MIN_REPEAT_STEPS


def test_dump_sample_is_fixed_and_fits_the_budget():
    import bench
    assert np.array_equal(bench.dump_sample(100, 1000, 5), np.arange(100))
    a, b = bench.dump_sample(32768, 6000, 21), bench.dump_sample(32768, 6000, 21)
    assert np.array_equal(a, b) and np.all(np.diff(a) > 0) and a[-1] < 32768
    assert len(a) * 6000 + 128 * 21 <= bench.DUMP_BYTES < (len(a) + 1) * 6000 + 128 * 21


def test_reference_arm_dump_is_reproducible(tmp_path):
    outs = []
    for run in ('a', 'b'):
        d = tmp_path / run
        subprocess.check_call([sys.executable, os.path.join(parity.ROOT, 'bench.py'), '--impl', 'reference', '--steps', '3',
                               '--warmup', '1', '--preroll', '2', '--dump-outputs', str(d)], stdout=subprocess.DEVNULL)
        outs.append({f: np.load(d / f) for f in sorted(os.listdir(d))})
    assert sorted(outs[0]) == ['dones.npy', 'env_index.npy', 'rewards.npy']
    for f, v in outs[0].items():
        assert v.dtype == np.float32 and np.array_equal(v, outs[1][f]), f
    assert outs[0]['rewards.npy'].shape == (4096, 4) and outs[0]['dones.npy'].shape == (4096,)
