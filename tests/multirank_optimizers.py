#!/usr/bin/env python
"""Momentum, Adagrad and RMSProp through the cross-process PS round
(``engine.TorchrunCluster`` under torchrun, world >= 2) against the C
restatement in tests/optimizer_oracle.c -- the companion of
tests/multirank_parity.py (SGD / Adam), whose gradient generator it reuses.

    python -m torch.distributed.run --nnodes=1 --nproc-per-node W \\
        --master-addr 127.0.0.1 --master-port P tests/multirank_optimizers.py \\
        [--cases small,nvls] [--rounds 3]

Rank r runs on GPU ``LOCAL_RANK mod n_gpus`` (on a 1-GPU box every rank shares
GPU 0).  Every case compares every hosted shard's var, state arrays and
global_step, and every rank's pulled parameters, BIT FOR BIT -- except the NVLS
round at world > 2, where the switch adds the W gradient copies in its own order.
There the bar is rtol = atol = 2e-6, as for SGD in multirank_parity.py: none of
the three normalises a step by the gradient's own magnitude the way Adam does
(the Adagrad accumulator starts at initial_accumulator_value, the RMSProp mean
square at 1), so a one-ulp change of the reduced gradient moves the update by
about lr times that ulp.
"""
import argparse
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

from tests.multirank_parity import MLP, bits, grad_np, grad_torch, seed_of  # noqa: E402
from tests import optimizer_oracle as oo  # noqa: E402

F = np.float32
HYPER = {oo.MOMENTUM: (0.05, 0.9, 0.0, 0.0), oo.ADAGRAD: (0.05, 0.1, 0.0, 0.0),
         oo.RMSPROP: (0.01, 0.9, 0.5, 1e-10)}


class Case(object):
    def __init__(self, name, opt, path="fused", wire="f32", mode="sum", entry="round", rtol=0.0):
        self.__dict__.update(locals())
        del self.__dict__["self"]


def build_cases(which, world):
    cases = []
    for opt in oo.OPTS:
        on = oo.NAMES[opt]
        if "small" in which:
            for path in ("fused", "staged"):
                for wire in ("f32", "bf16"):
                    for mode in ("sum", "mean", "async"):
                        cases.append(Case("%s/%s/%s/%s/round" % (on, path, wire, mode), opt,
                                          path=path, wire=wire, mode=mode))
            cases.append(Case("%s/fused/f32/async/graph" % on, opt, mode="async", entry="graph"))
        if "nvls" in which:
            tol = 0.0 if world <= 2 else 2e-6
            cases.append(Case("%s/nvls/f32/sum/round" % on, opt, path="nvls", rtol=tol))
            cases.append(Case("%s/nvls/f32/mean/graph" % on, opt, path="nvls", mode="mean",
                              entry="graph", rtol=tol))
    return cases


def make_optimizer(opt):
    from tfmesos_b200 import engine
    h = HYPER[opt]
    if opt == oo.MOMENTUM:
        return engine.MomentumOptimizer(h[0], h[1])
    if opt == oo.ADAGRAD:
        return engine.AdagradOptimizer(h[0], h[1])
    return engine.RMSPropOptimizer(*h)


def run_case(case, rounds, rank, world, device, dist):
    import torch
    from oracle import ps_oracle as o
    from tfmesos_b200 import engine, psx

    modes = {"sum": (psx.MODE_SUM, oo.SUM), "mean": (psx.MODE_SYNC_MEAN, oo.SYNC_MEAN),
             "async": (psx.MODE_ASYNC_ORDERED, oo.ASYNC_ORDERED)}
    pmode, omode = modes[case.mode]
    wire = psx.BF16 if case.wire == "bf16" else psx.F32
    cl = engine.TorchrunCluster(MLP, 1, make_optimizer(case.opt), wire=wire, device=device,
                                path=case.path)
    W = cl.n_workers
    dev = torch.device("cuda", device)
    wk, ws = cl.worker, cl.worker_stream
    tdt = torch.bfloat16 if wire == psx.BF16 else torch.float32

    refs = {}
    for key, ps in cl.servers.items():
        sp = ps.spec
        ref = oo.CShard(sp.nelem, case.opt, HYPER[case.opt])
        ref.var[:] = grad_np(sp.off, sp.off + sp.nelem, 777 + sp.task) * F(5.0)
        ps.shard.set_values(psx.VAR, ref.var)
        refs[key] = ref
    cl.barrier()

    def fill(rnd):
        if wk is None:
            return
        for t in range(cl.layout.ps_tasks):
            n = wk.grad_flat[t].numel()
            with torch.cuda.stream(ws):
                wk.grad_flat[t].copy_(grad_torch(n, seed_of(wk.index, rnd, t), dev).to(tdt))

    graph = None
    if case.entry == "graph":
        fill(0)
        graph = cl.capture_round(pmode)
    for rnd in range(1, rounds + 1):
        fill(rnd)
        if graph is not None:
            with torch.cuda.stream(ws):
                graph.replay()
        else:
            cl.round(pmode)
        for key, ps in cl.servers.items():
            sp = ps.spec
            slots = np.empty((W, sp.nelem), F)
            for w in range(W):
                g = grad_np(sp.off, sp.off + sp.nelem, seed_of(w, rnd, sp.task))
                slots[w] = o.bf16_to_f32(o.f32_to_bf16(g)) if wire == psx.BF16 else g
            refs[key].round(slots, omode)
    cl.barrier()
    if ws is not None:
        ws.synchronize()

    errors = []

    def same(got, want, what):
        if case.rtol == 0.0:
            if not np.array_equal(bits(got), bits(want)):
                bad = np.flatnonzero(bits(got) != bits(want))
                errors.append("%s: %d of %d elements differ (first %d: %r vs %r)"
                              % (what, bad.size, want.size, bad[0], got[bad[0]], want[bad[0]]))
        elif not np.allclose(got, want, rtol=case.rtol, atol=case.rtol):
            d = np.abs(got.astype(np.float64) - want)
            errors.append("%s: max abs diff %g (rtol %g)" % (what, float(d.max()), case.rtol))

    owned = {}
    for key, ps in cl.servers.items():
        ref = refs[key]
        same(ps.shard.get_values(psx.VAR), ref.var, "shard %r var" % (key,))
        same(ps.shard.get_values(psx.M), ref.m, "shard %r m" % (key,))
        if oo.STATE_ARRAYS[case.opt] == 2:
            same(ps.shard.get_values(psx.V), ref.v, "shard %r v" % (key,))
        want_step = rounds * (W if case.mode == "async" else 1)
        st = ps.shard.state()
        if st["global_step"] != want_step or ref.step != want_step:
            errors.append("shard %r global_step %d, oracle %d, expected %d"
                          % (key, st["global_step"], ref.step, want_step))
        owned[key] = o.f32_to_bf16(ref.var) if wire == psx.BF16 else ref.var
    # every rank checks its pulled parameters against the owners' oracle values
    table = [None] * world
    dist.all_gather_object(table, owned)
    want_all = {}
    for d in table:
        want_all.update(d)
    if wk is not None:
        for sp in cl.topo.shards:
            got = wk.param_flat[sp.task][sp.off:sp.off + sp.nelem]
            got = (got.view(torch.int16) if wire == psx.BF16 else got).cpu().numpy()
            if wire == psx.BF16:
                got = got.view(np.uint16)
                if case.rtol == 0.0:
                    same(got, want_all[sp.key], "pulled params of shard %r" % (sp.key,))
                else:
                    same(o.bf16_to_f32(got), o.bf16_to_f32(want_all[sp.key]),
                         "pulled params of shard %r" % (sp.key,))
            else:
                same(got, want_all[sp.key], "pulled params of shard %r" % (sp.key,))
    cl.close()
    return errors


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--cases", default="small")
    ap.add_argument("--rounds", type=int, default=3)
    args = ap.parse_args()
    import torch
    import torch.distributed as dist
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    n_gpus = torch.cuda.device_count()
    assert n_gpus >= 1, "multirank_optimizers needs a CUDA device: there is no CPU fallback"
    device = local % n_gpus
    torch.cuda.set_device(device)
    os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
    dist.init_process_group("gloo")
    failed = 0
    for case in build_cases(set(args.cases.split(",")), world):
        t0 = time.time()
        try:
            errors = run_case(case, args.rounds, rank, world, device, dist)
        except Exception as exc:                       # keep the other ranks in step
            import traceback
            errors = ["exception: %s\n%s" % (exc, traceback.format_exc())]
        flag = torch.tensor([1 if errors else 0])
        dist.all_reduce(flag)
        for e in errors:
            print("[rank %d] %s: %s" % (rank, case.name, e), flush=True)
        if rank == 0:
            print("CASE %-40s world=%d gpus=%d %s (%.1fs)"
                  % (case.name, world, min(world, n_gpus), "FAIL" if flag.item() else "ok",
                     time.time() - t0), flush=True)
        failed += int(flag.item() > 0)
        if errors and any(e.startswith("exception") for e in errors):
            break                                      # state after an exception is unknown
    dist.barrier()
    dist.destroy_process_group()
    if rank == 0:
        print("MULTIRANK OPTIMIZERS: %s" % ("FAILED (%d cases)" % failed if failed else "all ok"),
              flush=True)
    sys.exit(1 if failed else 0)


if __name__ == "__main__":
    main()
