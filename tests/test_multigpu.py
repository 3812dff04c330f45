"""Multi-GPU correctness as -m gpu tests: each runs one of the torchrun check scripts on 2 GPUs of this box and is skipped
when the box has fewer (the driver's single-GPU tiers).  tests/dp_nccl_check.py: N ranks on shards walk the trajectory of
one rank on the full batch (NCCL bucket, g_R over the peer ring, fused Adam, the NCCL-free step with the bucket in peer memory,
and that step captured as a CUDA graph on every rank).  tests/peer_check.py: g_R summed over NVLink peer memory inside the
backward (beside the g_R product from 8192 product rows, behind it below) == NCCL all-reduce of the partials, bit-identical
on every rank, buffers reused over steps; ranges of a PeerBucket summed in place == NCCL."""
import os
import socket
import subprocess
import sys

import pytest
import torch

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _torchrun(script, nproc=2, env=None, timeout=300):
    if torch.cuda.device_count() < nproc:
        pytest.skip(f"needs {nproc} GPUs, this box has {torch.cuda.device_count()}")
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        port = s.getsockname()[1]
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={nproc}", "--master-addr", "127.0.0.1",
           "--master-port", str(port), os.path.join(ROOT, "tests", script)]
    # a rank that never arrives must fail the test within its timeout, not hang the box: flag waits give up after 30 s
    r = subprocess.run(cmd, cwd=ROOT, env={"MPVAE_PEER_TIMEOUT_S": "30", **os.environ, **(env or {})}, capture_output=True,
                       text=True, timeout=timeout)
    sys.stdout.write(r.stdout[-4000:])
    sys.stderr.write(r.stderr[-2000:])
    return r


def test_data_parallel_step_matches_single_rank():
    r = _torchrun("dp_nccl_check.py")
    assert r.returncode == 0 and "DP_NCCL_CHECK PASS" in r.stdout


def test_peer_ring_equals_nccl_allreduce():
    r = _torchrun("peer_check.py")
    assert r.returncode == 0 and "PEER_CHECK PASS" in r.stdout


def test_serial_exchange_equals_nccl_allreduce():
    """MPVAE_FLAG_SERIAL_EXCHANGE: the stand-alone reduce kernel after the product at every shape."""
    r = _torchrun("peer_check.py", env={"PEER_CHECK_SERIAL": "1"})
    assert r.returncode == 0 and "PEER_CHECK PASS" in r.stdout
