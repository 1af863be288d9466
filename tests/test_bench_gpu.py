"""bench.py --dump-outputs: the files a run writes, their dtypes and size bound, and that a second run with the same arguments
writes the same outputs (so two builds can be compared file by file)."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
pytestmark = pytest.mark.gpu

ARGS = ['--gpus', '1', '--steps', '3', '--warmup', '1', '--size', '256', '--global-batch', '2', '--no-cpu-baseline',
        '--no-gpu-eager']
FILES = ['feature_l2', 'features_0', 'features_1', 'features_2', 'features_3', 'gate_loss', 'grad_l2', 'grads', 'step_loss']


def _bench(out):
    r = subprocess.run([sys.executable, os.path.join(ROOT, 'bench.py'), *ARGS, '--dump-outputs', str(out)],
                       capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stderr[-4000:]
    return json.loads(r.stdout.strip().splitlines()[-1])


def test_dump_outputs_repeat_across_runs(tmp_path):
    a, b = tmp_path / 'a', tmp_path / 'b'
    line = _bench(a)
    assert line['steps'] == 3
    _bench(b)
    assert sorted(os.listdir(a)) == sorted(os.listdir(b)) == sorted(f + '.npy' for f in FILES)
    assert sum(os.path.getsize(a / f) for f in os.listdir(a)) <= 64 << 20
    for f in FILES:
        x, y = np.load(a / f'{f}.npy'), np.load(b / f'{f}.npy')
        assert x.dtype in (np.float32, np.float64) and x.shape == y.shape and x.size > 0, f
        assert np.isfinite(x).all(), f
        # gradients accumulate with atomics, whose order differs between runs (tests/test_graph_gpu.py)
        assert np.abs(x - y).max() <= 5e-4 * np.abs(y).max(), f
