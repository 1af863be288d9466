"""Expert-parallel MoE over NVLink peer memory (BASELINE config 4 mechanism) on >= 2 GPUs of one box."""
import os
import subprocess
import sys

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
pytestmark = pytest.mark.gpu


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason='needs >= 2 GPUs')
def test_expert_parallel_matches_local_experts():
    n = 2
    r = subprocess.run([sys.executable, '-m', 'torch.distributed.run', '--nnodes=1', '--nproc-per-node', str(n),
                        '--master-addr', '127.0.0.1', '--master-port', '29543',
                        os.path.join(ROOT, 'tests', 'multi_gpu', 'ep_gpu_worker.py'), ROOT],
                       capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout[-4000:] + r.stderr[-4000:]
    assert r.stdout.count('ep ok noisy=False') == n, r.stdout[-2000:]
    assert r.stdout.count('ep ok noisy=True') == n, r.stdout[-2000:]
