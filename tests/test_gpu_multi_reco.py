"""GPU (-m gpu, needs >= 2 visible GPUs, skips otherwise): Recognition on template-sharded pipes under torch.distributed.run, one process
per GPU (sharded.NativeShardedPipe, symmetric-memory exchange buffers).  Every rank must return a single handle's results, frame after
frame.  The worker is tools/check_multi_gpu_reco.py."""
import os
import subprocess
import sys

import pytest

from test_gpu_multi import ROOT, _free_port, _n_gpus

pytestmark = pytest.mark.gpu


@pytest.mark.parametrize("world", [2, 4, 8])
def test_sharded_recognition_parity_under_torchrun(world):
    n = _n_gpus()
    if n < world:
        pytest.skip("%d GPU(s) visible, the test needs %d" % (n, world))
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", str(world), "--master-addr", "127.0.0.1",
           "--master-port", str(_free_port()), os.path.join(ROOT, "tools", "check_multi_gpu_reco.py")]
    r = subprocess.run(cmd, cwd=ROOT, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, timeout=600)
    tail = r.stdout[-3000:]
    assert r.returncode == 0, tail
    assert "MULTI-GPU RECO PARITY PASS" in r.stdout, tail
