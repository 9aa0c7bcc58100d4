"""Checkpoint / restore of PS shards (SURVEY.md 8f-4), standing in for what the
reference gets from ``tf.train.Supervisor(logdir=...)`` (TF checkpoints written
by the chief, examples/mnist/mnist_replica.py:165-170).

One safetensors file per process: every hosted stripe's ``var`` (+ the
optimizer's state arrays ``m`` [, ``v``]) as float32 tensors keyed ``<region>/ps<task>/stripe<j>``, and the scalars
(global_step, stored beta powers) in the metadata.  Restoring puts back exactly
those bits, so a resumed run continues bit-identically (tests/test_gpu_checkpoint.py).
"""
import json
import os

from . import psx


def _regions(ps):
    n_state = psx.OPT_STATE_ARRAYS[ps.shard.opt]
    return [("var", psx.VAR), ("m", psx.M), ("v", psx.V)][:1 + n_state]


def shard_file(path, rank=0, world=1):
    return "%s-%05d-of-%05d.safetensors" % (path, rank, world)


def save(cluster, path, rank=0, world=1):
    """cluster: anything with ``.servers`` ({(task, stripe): ParameterServer})."""
    from safetensors.numpy import save_file
    tensors, meta = {}, {}
    for (task, stripe), ps in cluster.servers.items():
        for name, which in _regions(ps):
            tensors["%s/ps%d/stripe%d" % (name, task, stripe)] = ps.shard.get_values(which)
        st = ps.shard.state()
        meta["state/ps%d/stripe%d" % (task, stripe)] = json.dumps(
            {"global_step": st["global_step"],
             # float32 values survive the round trip through repr exactly
             "beta1_power": repr(st["beta1_power"]), "beta2_power": repr(st["beta2_power"]),
             "nelem": ps.spec.nelem, "off": ps.spec.off, "opt": ps.shard.opt})
    fn = shard_file(path, rank, world)
    # write-then-rename (what TF's Saver does): a crash during save never destroys
    # the previous checkpoint
    save_file(tensors, fn + ".tmp", metadata=meta)
    os.replace(fn + ".tmp", fn)
    return fn


def restore(cluster, path, rank=0, world=1):
    from safetensors import safe_open
    fn = shard_file(path, rank, world)
    with safe_open(fn, framework="numpy") as f:
        meta = f.metadata()
        for (task, stripe), ps in cluster.servers.items():
            st = json.loads(meta["state/ps%d/stripe%d" % (task, stripe)])
            if st["nelem"] != ps.spec.nelem or st["off"] != ps.spec.off or st["opt"] != ps.shard.opt:
                raise RuntimeError("checkpoint %s does not match shard ps%d/stripe%d "
                                   "(layout or optimizer changed)" % (fn, task, stripe))
            for name, which in _regions(ps):
                ps.shard.set_values(which, f.get_tensor("%s/ps%d/stripe%d" % (name, task, stripe)))
            ps.shard.set_state(float(st["beta1_power"]), float(st["beta2_power"]),
                               st["global_step"])
    return fn
