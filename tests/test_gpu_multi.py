"""GPU (>= 2 devices): the data-parallel learner equals the single-GPU full-batch learner and the
float64 oracle, with the gradient exchange as a push over NVLink peer memory from the backward's
tail (default), from the stand-alone producer kernel, and through NCCL."""
import os
import socket
import subprocess
import sys

import pytest
import torch

pytestmark = pytest.mark.gpu


@pytest.mark.parametrize("allreduce", ["peer", "peer-standalone", "nccl"])
def test_two_rank_learner_matches_single_gpu(allreduce):
    if torch.cuda.device_count() < 2:
        pytest.skip("needs at least 2 GPUs")
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        port = s.getsockname()[1]
    script = os.path.join(os.path.dirname(__file__), "multi_gpu_check.py")
    res = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2",
                          "--master-addr", "127.0.0.1", "--master-port", str(port), script],
                         capture_output=True, text=True, timeout=240,
                         env=dict(os.environ, IMPALA_ALLREDUCE=allreduce.split("-")[0],
                                  IMPALA_PUSH_FUSED="0" if allreduce == "peer-standalone" else "1"))
    assert res.returncode == 0, res.stdout[-3000:] + res.stderr[-3000:]
    assert "MULTI_GPU_OK" in res.stdout
    want = {"peer": "allreduce=peer(fused)", "peer-standalone": "allreduce=peer(standalone)", "nccl": "allreduce=nccl"}[allreduce]
    assert want in res.stdout  # the requested path is the one that ran


@pytest.mark.parametrize("transport", ["queue", "ring"])
def test_dp_learner_process_two_gpus(tmp_path, transport):
    """SURVEY 8e through the PRODUCT API: one forked `Learner(devices=[cuda:0, cuda:1])` behind the
    real queue / ring, worker rank spawned by it, shards DMA'd per rank, weights compared with the
    real reference's (golden c1)."""
    if torch.cuda.device_count() < 2:
        pytest.skip("needs at least 2 GPUs")
    script = os.path.join(os.path.dirname(__file__), "learner_process_check.py")
    res = subprocess.run([sys.executable, script, str(tmp_path / "logs"), transport, "2"], capture_output=True,
                         text=True, timeout=300)
    assert res.returncode == 0, res.stdout[-3000:] + res.stderr[-3000:]
    assert "LEARNER_PROCESS_OK" in res.stdout and "devices=2" in res.stdout
