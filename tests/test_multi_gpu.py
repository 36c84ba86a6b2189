"""Multi-GPU data path on real devices (needs >= 2 GPUs; skipped on a 1-GPU box): torchrun with
2 ranks runs tools/dist_check.py -- shared-frame (NVLink peer stores, fused resolve+gather) and
NCCL-gather frames must both be bit-identical to the 1-rank frame, in PATH and REF mode."""
import os
import socket
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.mark.gpu
def test_two_ranks_bit_identical_to_one():
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs (tools/dist_check.py under torchrun with 2 ranks; profiles/README.md)")
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2",
                        "--master-addr", "127.0.0.1", "--master-port", str(port),
                        os.path.join(ROOT, "tools", "dist_check.py")], capture_output=True, text=True, timeout=600)
    print(r.stdout[-3000:])
    assert r.returncode == 0, r.stderr[-3000:]
    assert "dist_check: OK" in r.stdout
