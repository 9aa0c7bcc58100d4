"""Momentum, Adagrad and RMSProp through the cross-process ``TorchrunCluster``
round, bit for bit against the C restatement (tests/multirank_optimizers.py does
the work; this file launches it under torchrun).

On a 1-GPU box the ranks share GPU 0; with >= 2 GPUs and NVSwitch multicast the
``multigpu`` case adds the NVLS round (bit-exact at world 2, rtol 2e-6 beyond --
the harness's docstring says why).
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


def _launch(world, cases, timeout):
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1",
           "--nproc-per-node", str(world), "--master-addr", "127.0.0.1",
           "--master-port", str(_free_port()),
           os.path.join(ROOT, "tests", "multirank_optimizers.py"), "--cases", cases]
    env = dict(os.environ, PYTHONUNBUFFERED="1", OMP_NUM_THREADS="4")
    p = subprocess.run(cmd, cwd=ROOT, env=env, stdout=subprocess.PIPE, stderr=subprocess.STDOUT,
                       text=True, timeout=timeout)
    lines = p.stdout.splitlines()
    verdicts = [l for l in lines if l.startswith(("CASE", "[rank", "MULTIRANK"))]
    tail = "\n".join(verdicts[-60:] + ["..."] + lines[-20:])
    assert p.returncode == 0, "multirank optimizers failed (world %d, %s):\n%s" % (world, cases,
                                                                                 tail)
    assert "MULTIRANK OPTIMIZERS: all ok" in p.stdout, tail
    return p.stdout


@pytest.mark.timeout(900)
@pytest.mark.parametrize("world", [2, 4])
def test_fused_and_staged_rounds_bit_exact(world):
    """fused and staged x f32 and bf16 x sum / mean / async, and a captured-graph
    round, for each of the three optimizers: shards and pulled parameters."""
    out = _launch(world, "small", timeout=850)
    for name in ("momentum", "adagrad", "rmsprop"):
        assert "%s/fused/f32/async/graph" % name in out


@pytest.mark.multigpu
@pytest.mark.timeout(900)
def test_nvls_round_one_rank_per_gpu():
    import torch
    from tfmesos_b200 import psx
    world = min(torch.cuda.device_count(), 8)
    if world < 2 or not all(psx.nvls_supported(d) for d in range(world)):
        pytest.skip("needs >= 2 GPUs with NVSwitch multicast")
    _launch(world, "nvls", timeout=850)
