"""Multi-GPU parity (needs >= 2 GPUs on the box; skipped otherwise): every data-parallel path of the library against the
2-rank run of the unmodified reference (tests/golden/update_ppolag_parallel2.npz).  See tools/mgpu_parity.py."""
import os
import subprocess
import sys

import pytest
import torch

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.mark.timeout(600)
def test_two_rank_parity_all_paths():
    if torch.cuda.device_count() < 2:
        pytest.skip('needs 2 GPUs (on a machine with two or more: python -m pytest tests/test_multigpu_gpu.py -m gpu)')
    cmd = [sys.executable, '-m', 'torch.distributed.run', '--nnodes=1', '--nproc-per-node', '2', '--master-addr', '127.0.0.1',
           '--master-port', '29541', os.path.join(ROOT, 'tools', 'mgpu_parity.py')]
    out = subprocess.run(cmd, capture_output=True, text=True, timeout=500, cwd=ROOT)
    print(out.stdout[-4000:])
    assert out.returncode == 0 and 'MULTI-RANK PARITY OK' in out.stdout, out.stdout[-3000:] + out.stderr[-3000:]
