"""2-GPU parity (skips with < 2 GPUs): the NCCL weight-distribution paths of the WeightStreamer, checked on EVERY rank against the
reference's output (stored under tests/golden/) -- rank 0 is the root that never receives data, so rank 1's output is the one that proves the collective."""
import os
import subprocess
import sys
import tempfile

import pytest

from onnxstream_b200 import emit

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _ngpus():
    try:
        import torch
        return torch.cuda.device_count()
    except Exception:
        return 0


@pytest.mark.skipif(_ngpus() < 2, reason="needs 2 GPUs")
@pytest.mark.parametrize("sharded", ["1", "0"])
def test_two_ranks_match_reference(sharded):
    with tempfile.TemporaryDirectory(prefix="osb200_mgpu_") as tmp:
        d = tmp + "/"
        emit.emit_unet(d, emit.UNetConfig.tiny(16), "float16", seed=0)
        env = dict(os.environ, OSB_SHARDED_H2D=sharded)
        env.pop("CUDA_VISIBLE_DEVICES", None)
        cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr", "127.0.0.1", "--master-port", "29613",
               os.path.join(ROOT, "tests", "mgpu_worker.py"), d]
        r = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, timeout=600, env=env)
        lines = [l for l in r.stdout.splitlines() if l.startswith("MGPU_")]
        assert r.returncode == 0 and len(lines) == 2 and all(l.startswith("MGPU_OK") for l in lines), r.stdout[-3000:]
        assert any("rank 1/2" in l for l in lines)
