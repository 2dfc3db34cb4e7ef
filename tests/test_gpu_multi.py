"""On-GPU multi-rank correctness (needs >= 2 GPUs: `python -m pytest tests/test_gpu_multi.py -m gpu` on a machine with two).
The host-side N > 1 logic is also covered on CPU by tests/test_host_cpu.py::test_data_parallel_world2_gloo."""
import os
import subprocess
import sys

import pytest
import torch

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason='needs two GPUs')
def test_two_rank_gradients_and_parameters_on_gpu():
    port = 29500 + os.getpid() % 2000
    cmd = [sys.executable, '-m', 'torch.distributed.run', '--nnodes=1', '--nproc-per-node', '2', '--master-addr',
           '127.0.0.1', '--master-port', str(port), os.path.join(ROOT, 'tests', '_ddp_gpu_worker.py')]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=600, cwd=ROOT)
    sys.stdout.write(r.stdout[-3000:])
    sys.stderr.write(r.stderr[-3000:])
    assert r.returncode == 0 and 'DDP_CHECK OK' in r.stdout
