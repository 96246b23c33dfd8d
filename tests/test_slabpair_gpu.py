"""Multi-GPU pair slab run == single-GPU run, bit for bit, through torchrun (needs >= 2 GPUs): tools/slabpair_check.py."""
import os
import subprocess
import sys

import pytest

from helpers import ROOT

pytestmark = pytest.mark.gpu


def test_pair_slabs_match_single_gpu(built):
    import torch
    n = torch.cuda.device_count()
    if n < 2:
        pytest.skip("needs at least 2 GPUs")
    world = 2 if n < 4 else 4
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", str(world),
                        "--master-addr", "127.0.0.1", "--master-port", "29617", os.path.join(ROOT, "tools", "slabpair_check.py")],
                       stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, timeout=900)
    assert r.returncode == 0 and "SLABPAIR_CHECK_OK" in r.stdout, r.stdout[-3000:]
