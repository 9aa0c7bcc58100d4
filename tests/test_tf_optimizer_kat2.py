"""TensorFlow's own published known answers for Momentum, Adagrad and RMSProp
(momentum_test.py / adagrad_test.py / rmsprop_test.py, TF r0.12) held against
both CPU restatements and the CUDA kernels at TF's float32 tolerance.  The
vectors and their provenance: tests/golden/make_tf_optimizer_kat2.py."""
import json
import os

import numpy as np
import pytest

from tests import optimizer_oracle as oo

F = np.float32
KAT = json.load(open(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden",
                                  "tf_optimizer_kat2.json")))
RTOL, ATOL = KAT["tolerance"]["rtol"], KAT["tolerance"]["atol"]
INP = KAT["inputs"]
VAR = np.array(INP["var0"] + INP["var1"], F)       # one 4-element bucket: var0 | var1
GRAD = np.array(INP["grads0"] + INP["grads1"], F)


def cases():
    """(name, opt id, hyper, steps[{t, var0, var1, ...}])"""
    m, a = KAT["momentum"], KAT["adagrad"]
    out = [("momentum", oo.MOMENTUM, (m["learning_rate"], m["momentum"], 0.0, 0.0), m["steps"]),
           ("adagrad", oo.ADAGRAD, (a["learning_rate"], a["initial_accumulator_value"], 0.0, 0.0),
            a["steps"])]
    for r in KAT["rmsprop"]:
        out.append(("rmsprop_" + r["test"], oo.RMSPROP,
                    (r["learning_rate"], r["decay"], r["momentum"], r["epsilon"]), r["steps"]))
    return out


CASES = cases()


def _want(st):
    return np.array(st["var0"] + st["var1"], np.float64)


@pytest.mark.parametrize("cls", [oo.Shard, oo.CShard])
@pytest.mark.parametrize("name,opt,hyper,steps", CASES, ids=[c[0] for c in CASES])
def test_restatements_reproduce_tf_testbasic(cls, name, opt, hyper, steps):
    sh = cls(4, opt, hyper)
    sh.var[:] = VAR
    t = 0
    for st in steps:
        while t < st["t"]:
            sh.round(GRAD[None, :], oo.SUM)
            t += 1
        np.testing.assert_allclose(sh.var, _want(st), rtol=RTOL, atol=ATOL)
        if "accum0" in st:
            np.testing.assert_allclose(sh.m[:2], st["accum0"], rtol=RTOL, atol=ATOL)
        if "rms0" in st:
            np.testing.assert_allclose(sh.m[:2], st["rms0"], rtol=RTOL, atol=ATOL)
            np.testing.assert_allclose(sh.v[:2], st["mom0"], rtol=RTOL, atol=ATOL)
    assert sh.step == t


@pytest.mark.gpu
@pytest.mark.parametrize("fused", [False, True])
def test_cuda_kernels_reproduce_tf_testbasic(fused):
    """The same vectors through libpsx.so: push -> apply -> pull, and psx_round."""
    import torch
    from tfmesos_b200 import engine, psx
    psx.init(0)
    for name, opt, hyper, steps in CASES:
        optimizer = {oo.MOMENTUM: lambda h: engine.MomentumOptimizer(h[0], h[1]),
                     oo.ADAGRAD: lambda h: engine.AdagradOptimizer(h[0], h[1]),
                     oo.RMSPROP: lambda h: engine.RMSPropOptimizer(*h)}[opt](hyper)
        cl = engine.LocalCluster([("v", (4,))], 1, 1, optimizer, fused=fused)
        try:
            cl.set_variable("v", VAR)
            cl.workers[0].grads["v"].copy_(torch.from_numpy(GRAD))
            t = 0
            for st in steps:
                while t < st["t"]:
                    cl.round(psx.MODE_SUM)
                    t += 1
                torch.cuda.synchronize()
                np.testing.assert_allclose(cl.get_variable("v"), _want(st), rtol=RTOL, atol=ATOL,
                                           err_msg=name)
                np.testing.assert_allclose(cl.workers[0].params["v"].cpu().numpy(), _want(st),
                                           rtol=RTOL, atol=ATOL, err_msg=name)
            assert cl.global_step() == t
        finally:
            cl.close()
