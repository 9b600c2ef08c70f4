"""2-GPU check of the partitioned layer and the entity-sharded scorer (skipped on a 1-GPU box)."""
import os
import socket
import subprocess
import sys

import pytest
import torch

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_two_gpu_partitioned_layer_and_sharded_rank():
    if torch.cuda.device_count() < 2:
        pytest.skip('needs 2 GPUs')
    s = socket.socket()
    s.bind(('127.0.0.1', 0))
    port = s.getsockname()[1]
    s.close()
    cmd = [sys.executable, '-m', 'torch.distributed.run', '--nnodes=1', '--nproc-per-node', '2', '--master-addr', '127.0.0.1',
           '--master-port', str(port), os.path.join(ROOT, 'tests', 'dist_gpu_check.py')]
    p = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, timeout=600)
    assert p.returncode == 0 and 'DIST_OK' in p.stdout, p.stdout[-4000:]
