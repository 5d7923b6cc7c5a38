"""Multi-GPU tier of training checkpoints: spawns scripts/checkpoint_resume_check.py under torch.distributed.run over
EVERY visible GPU (skipped below 2 GPUs), and with two ranks sharing one GPU.  A training state saved by the one-GPU
interactive trainer resumes sharded, and one saved sharded resumes on one GPU; both must end bit-identical (weights,
AdamW state, losses) to the uninterrupted one-GPU run, on every rank."""
import os
import socket
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _check(ranks, gpus):
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        port = s.getsockname()[1]
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", str(ranks), "--master-addr",
           "127.0.0.1", "--master-port", str(port), os.path.join(ROOT, "scripts", "checkpoint_resume_check.py")]
    env = dict(os.environ)
    if gpus == 1:        # the first visible GPU only: the ranks share it
        env["CUDA_VISIBLE_DEVICES"] = os.environ.get("CUDA_VISIBLE_DEVICES", "0").split(",")[0]
    r = subprocess.run(cmd, cwd=ROOT, capture_output=True, text=True, timeout=900, env=env)
    print(r.stdout[-3000:])
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
    assert "checkpoint_resume_check world=%d gpus=%d: OK" % (ranks, gpus) in r.stdout, r.stdout[-3000:]


@pytest.mark.gpu
def test_resume_across_world_sizes():
    import torch
    n = torch.cuda.device_count()
    if n < 2:
        pytest.skip("needs >= 2 GPUs (found %d)" % n)
    _check(n, n)


@pytest.mark.gpu
def test_resume_across_world_sizes_two_ranks_on_one_gpu():
    _check(2, 1)
