"""Multi-GPU tier of bf16 interactive training: scripts/interactive_train_check.py --precision 1 under
torch.distributed.run at world size 2, on two GPUs (skipped below 2 GPUs) and with the two ranks sharing one GPU.  After 3
iterations of dist.train_interactive_sharded(..., precision=1) the weights of every rank must be bit-identical to each
other and to train.train_interactive(..., precision=1) on one GPU, for the cases the script covers."""
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
           "127.0.0.1", "--master-port", str(port), os.path.join(ROOT, "scripts", "interactive_train_check.py"),
           "--precision", "1"]
    env = dict(os.environ)
    if gpus == 1:        # the first visible GPU only: the ranks share it
        env["CUDA_VISIBLE_DEVICES"] = os.environ.get("CUDA_VISIBLE_DEVICES", "0").split(",")[0]
    r = subprocess.run(cmd, cwd=ROOT, capture_output=True, text=True, timeout=900, env=env)
    print(r.stdout[-3000:])
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
    assert "training precision 1" in r.stdout, r.stdout[-3000:]
    assert "interactive_train_check world=%d gpus=%d: OK" % (ranks, gpus) in r.stdout, r.stdout[-3000:]


@pytest.mark.gpu
def test_sharded_bf16_weights_equal_the_single_gpu_run():
    import torch
    n = torch.cuda.device_count()
    if n < 2:
        pytest.skip("needs >= 2 GPUs (found %d)" % n)
    _check(2, 2)


@pytest.mark.gpu
def test_two_ranks_on_one_gpu_bf16():
    _check(2, 1)
