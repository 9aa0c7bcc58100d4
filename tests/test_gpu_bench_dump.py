"""bench.py --dump-outputs writes what the timed round computed: the parameters
worker 0 pulled in the last timed step, bit for bit what the oracle gets by
replaying the same rounds on the same synthetic gradients."""
import importlib.util
import json
import os
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _bench_module():
    spec = importlib.util.spec_from_file_location("bench_mod", os.path.join(ROOT, "bench.py"))
    bench = importlib.util.module_from_spec(spec)
    sys.modules["bench_mod"] = bench
    spec.loader.exec_module(bench)
    return bench


@pytest.mark.timeout(600)
def test_dump_outputs_are_the_pulled_parameters_of_the_last_step(tmp_path):
    """The 25.6e6-element bucket exceeds the dump budget, so this also pins the
    sampled positions (bench.dump_index)."""
    steps, warmup = 4, 3
    cmd = [sys.executable, os.path.join(ROOT, "bench.py"), "--workload", "resnet50_bucket",
           "--steps", str(steps), "--warmup", str(warmup), "--no-e2e", "--no-staged",
           "--no-mnist", "--no-cpu-baseline", "--dump-outputs", str(tmp_path)]
    p = subprocess.run(cmd, cwd=ROOT, stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True,
                       timeout=550)
    assert p.returncode == 0, p.stderr[-3000:]
    line = json.loads([l for l in p.stdout.splitlines() if l.startswith("{")][-1])
    assert line["steps"] == steps and line["warmup"] == warmup and line["verified"] is True

    assert sorted(os.listdir(tmp_path)) == ["flat.npy"]
    assert os.path.getsize(tmp_path / "flat.npy") <= 64 << 20
    got = np.load(tmp_path / "flat.npy")
    bench = _bench_module()
    idx = bench.dump_index(bench.n_params("resnet50_bucket"), 1)
    assert idx is not None and got.dtype == np.float32 and got.shape == idx.shape

    from oracle import ps_oracle as o
    ref = o.CShard(idx.size, o.ADAM, lr=0.01)
    slots = bench.synth_np(idx, bench.grad_seed(0, 0))[None]
    for _ in range(warmup + steps):
        ref.round(slots, o.SUM)
    assert np.array_equal(got.view(np.uint32), ref.var.view(np.uint32))
