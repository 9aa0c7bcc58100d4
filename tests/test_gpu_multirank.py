"""The configuration SCALE measures -- cross-process ``TorchrunCluster`` under
torchrun, world >= 2 -- checked bit for bit against the oracle
(tests/multirank_parity.py does the work; this file launches it).

On a 1-GPU box the ranks share GPU 0 (CUDA IPC between processes on one device:
same kernels, same protocol, no NVLink); with >= 2 GPUs the ``multigpu`` cases
run one rank per GPU up to 8 and add the NVLS round.
"""
import os
import socket
import subprocess
import sys

import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    return port


def _launch(world, cases, rounds=3, timeout=1100, only=None):
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1",
           "--nproc-per-node", str(world), "--master-addr", "127.0.0.1",
           "--master-port", str(_free_port()),
           os.path.join(ROOT, "tests", "multirank_parity.py"), "--cases", cases,
           "--rounds", str(rounds)]
    if only:
        cmd += ["--only", only]
    env = dict(os.environ, PYTHONUNBUFFERED="1", OMP_NUM_THREADS="4")
    p = subprocess.run(cmd, cwd=ROOT, env=env, stdout=subprocess.PIPE, stderr=subprocess.STDOUT,
                       text=True, timeout=timeout)
    # the per-case verdicts and every rank's errors first: torchrun's own report of
    # the failed children fills the end of the output
    lines = p.stdout.splitlines()
    verdicts = [l for l in lines if l.startswith(("CASE", "[rank", "MULTIRANK"))]
    tail = "\n".join(verdicts[-60:] + ["..."] + lines[-20:])
    assert p.returncode == 0, "multirank parity failed (world %d, %s):\n%s" % (world, cases, tail)
    assert "MULTIRANK PARITY: all ok" in p.stdout, tail
    return p.stdout


def _n_gpus():
    import torch
    return torch.cuda.device_count()


@pytest.mark.timeout(1200)
def test_world2_small_and_full_size_bit_exact():
    """2 ranks: every path x wire x discipline on the MNIST-replica bucket, and the
    full 2.0e8-element NMF parameter set through the fused round (SCALE's
    headline) and round_host (its e2e) -- shards and pulled parameters equal the
    oracle bit for bit."""
    out = _launch(2, "small,fullmin")
    assert "nmf/fused/f32/sum/round" in out and "round_host" in out


@pytest.mark.timeout(900)
def test_world4_small_bit_exact():
    """4 ranks incl. PS shards on ranks that host no worker (dedicated PS GPUs)."""
    out = _launch(4, "small", timeout=850)
    assert "dedicated-ps" in out


@pytest.mark.multigpu
@pytest.mark.timeout(1500)
def test_one_rank_per_gpu_up_to_8_full_size_and_nvls():
    """One rank per GPU over NVLink (world = min(n_gpus, 8)): small + full-size
    cases bit-exact; the NVLS round bit-exact at world 2, rtol 2e-6 beyond."""
    world = min(_n_gpus(), 8)
    from tfmesos_b200 import psx
    cases = "small,fullmin"
    if all(psx.nvls_supported(d) for d in range(world)):
        cases += ",nvls"
    _launch(world, cases, timeout=1400)
