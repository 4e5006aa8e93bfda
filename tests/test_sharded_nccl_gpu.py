"""Multi-rank `-m gpu` test (needs >= 2 GPUs, skipped otherwise): the gene-sharded device-resident pipeline over NCCL --
one rank per GPU, the global dispersion-trend step through one packed all-gather, ONE packed all-gather of the results
(sharded.PackedGather; R/parallel.R:25-28, 54-66) -- equals the single-GPU run bit for bit.  The same logic runs on CPU
with gloo and the emulated engine in tests/test_sharded_gloo.py."""
import os
import subprocess
import sys

import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_sharded_device_pipeline_over_nccl_equals_whole():
    import torch
    n_gpu = torch.cuda.device_count()
    if n_gpu < 2:
        pytest.skip("needs at least 2 GPUs")
    world = 4 if n_gpu >= 4 else 2
    env = dict(os.environ)
    for k in ("RANK", "WORLD_SIZE", "LOCAL_RANK", "MASTER_ADDR", "MASTER_PORT"):
        env.pop(k, None)
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={world}",
                        "--master-addr", "127.0.0.1", "--master-port", "29641",
                        os.path.join(ROOT, "scripts", "sharded_device_nccl.py")], env=env, capture_output=True, text=True,
                       timeout=600)
    assert r.returncode == 0, (r.stdout[-2000:], r.stderr[-3000:])
    assert "sharded == whole: True" in r.stdout and "per-gene collectives: 2" in r.stdout, r.stdout[-2000:]
