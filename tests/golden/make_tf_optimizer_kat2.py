#!/usr/bin/env python
"""Writes tests/golden/tf_optimizer_kat2.json: the known answers of TensorFlow's
own unit tests for the Momentum, Adagrad and RMSProp optimizers (TensorFlow
r0.12, tensorflow/python/training/), the companion of tf_optimizer_kat.json
(SGD, Adam).

All three tests use var0 = [1.0, 2.0], var1 = [3.0, 4.0], grads0 = [0.1, 0.1],
grads1 = [0.01, 0.01] (float32 leg) and compare through
assertAllCloseAccordingToType (float32: rtol = atol = 1e-6).

* ``momentum_test.py`` ``MomentumOptimizerTest.testBasic``:
  MomentumOptimizer(learning_rate=2.0, momentum=0.9), two steps.  After step 1
  the test asserts accum0 == [0.1, 0.1], var0 == [1.0 - 0.1 * 2.0, 2.0 - 0.1 * 2.0],
  var1 == [3.0 - 0.01 * 2.0, 4.0 - 0.01 * 2.0]; after step 2
  accum0 == [0.9 * 0.1 + 0.1, ...] and
  var0 == [1.0 - 0.1 * 2.0 - (0.9 * 0.1 + 0.1) * 2.0, ...].

* ``adagrad_test.py`` ``AdagradOptimizerTest.testBasic``:
  AdagradOptimizer(3.0, initial_accumulator_value=0.1), three steps; the test
  asserts var0 == [-1.6026098728179932, -0.6026098728179932] and
  var1 == [2.715679168701172, 3.715679168701172].

* ``rmsprop_test.py`` ``testWithoutMomentum``: RMSPropOptimizer(learning_rate=2.0,
  decay=0.9, momentum=0.0, epsilon=1.0), and ``testWithMomentum``: the same with
  momentum=0.5, epsilon=1e-5.  The ``rms`` slot starts at 1.0, ``momentum`` at 0;
  the tests spell each step out, e.g. after step 1 rms0 == [0.901, 0.901] and
  var0 == [1.0 - (0.1 * 2.0 / math.sqrt(0.901 + 1.0)), ...].

This script evaluates those published formulas step by step in float64 -- it
does NOT import any restatement of the PS data path -- and stores the expected
values; tests/test_tf_optimizer_kat2.py holds both CPU restatements and the CUDA
kernels to TF's own tolerance.  Adagrad's var is the test's literal constant.
"""
import json
import math
import os

import numpy as np

VAR0, VAR1 = [1.0, 2.0], [3.0, 4.0]
G0, G1 = [0.1, 0.1], [0.01, 0.01]


def f32(xs):
    """The float32 inputs of the test's float32 leg, as float64 values."""
    return [float(np.float32(x)) for x in xs]


def momentum_steps(lr, mu, steps):
    out = []
    v0, v1, a0, a1 = list(VAR0), list(VAR1), [0.0, 0.0], [0.0, 0.0]
    g0, g1 = f32(G0), f32(G1)
    for t in range(1, steps + 1):
        a0 = [a * mu + g for a, g in zip(a0, g0)]
        a1 = [a * mu + g for a, g in zip(a1, g1)]
        v0 = [v - a * lr for v, a in zip(v0, a0)]
        v1 = [v - a * lr for v, a in zip(v1, a1)]
        out.append({"t": t, "var0": v0, "var1": v1, "accum0": a0, "accum1": a1})
    return out


def rmsprop_steps(lr, decay, mu, eps, steps):
    out = []
    v0, v1 = list(VAR0), list(VAR1)
    r0, r1, m0, m1 = [1.0, 1.0], [1.0, 1.0], [0.0, 0.0], [0.0, 0.0]
    g0, g1 = f32(G0), f32(G1)
    for t in range(1, steps + 1):
        r0 = [r * decay + (1 - decay) * g * g for r, g in zip(r0, g0)]
        r1 = [r * decay + (1 - decay) * g * g for r, g in zip(r1, g1)]
        m0 = [m * mu + g * lr / math.sqrt(r + eps) for m, g, r in zip(m0, g0, r0)]
        m1 = [m * mu + g * lr / math.sqrt(r + eps) for m, g, r in zip(m1, g1, r1)]
        v0 = [v - m for v, m in zip(v0, m0)]
        v1 = [v - m for v, m in zip(v1, m1)]
        out.append({"t": t, "var0": v0, "var1": v1, "rms0": r0, "mom0": m0})
    return out


def main():
    out = {"source": "tensorflow r0.12 python/training/{momentum,adagrad,rmsprop}_test.py",
           "tolerance": {"rtol": 1e-6, "atol": 1e-6,
                         "why": "assertAllCloseAccordingToType, float32 leg"},
           "inputs": {"var0": VAR0, "var1": VAR1, "grads0": f32(G0), "grads1": f32(G1)}}
    out["momentum"] = {"learning_rate": 2.0, "momentum": 0.9,
                       "steps": momentum_steps(2.0, 0.9, 2)}
    out["adagrad"] = {"learning_rate": 3.0, "initial_accumulator_value": 0.1,
                      "steps": [{"t": 3,
                                 "var0": [-1.6026098728179932, -0.6026098728179932],
                                 "var1": [2.715679168701172, 3.715679168701172]}]}
    out["rmsprop"] = [
        {"test": "testWithoutMomentum", "learning_rate": 2.0, "decay": 0.9, "momentum": 0.0,
         "epsilon": 1.0, "steps": rmsprop_steps(2.0, 0.9, 0.0, 1.0, 2)},
        {"test": "testWithMomentum", "learning_rate": 2.0, "decay": 0.9, "momentum": 0.5,
         "epsilon": 1e-5, "steps": rmsprop_steps(2.0, 0.9, 0.5, 1e-5, 2)},
    ]
    path = os.path.join(os.path.dirname(os.path.abspath(__file__)), "tf_optimizer_kat2.json")
    with open(path, "w") as f:
        json.dump(out, f, indent=1)
    print(path)


if __name__ == "__main__":
    main()
