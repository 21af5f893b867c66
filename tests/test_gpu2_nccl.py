"""Two-GPU NCCL run of `parallel.read_sharded` (markers ``gpu`` and
``gpu2``; `python -m pytest tests -m gpu2` on a machine with at least two
GPUs).  With fewer GPUs it is skipped; the world-size-2 logic is also
covered on CPU under gloo (tests/test_distributed_gloo.py)."""
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _ngpu():
    import torch
    return torch.cuda.device_count()


@pytest.mark.gpu
@pytest.mark.gpu2
@pytest.mark.skipif(_ngpu() < 2, reason='needs two GPUs')
def test_sharded_read_and_gather_nccl():
    res = subprocess.run(
        [sys.executable, '-m', 'torch.distributed.run', '--nnodes=1',
         '--nproc-per-node', '2', '--master-addr', '127.0.0.1',
         '--master-port', '29731', 'tests/check_nccl_gather.py'],
        cwd=ROOT, capture_output=True, text=True, timeout=600)
    assert res.returncode == 0, res.stdout + res.stderr
    assert 'nccl sharded read + gather on 2 GPUs: OK' in res.stdout, \
        res.stdout + res.stderr
