#!/usr/bin/env python
"""Oracle parity of the cross-process PS round, at the configuration bench.py /
SCALE measure: ``engine.TorchrunCluster`` under torchrun, world >= 2, one process
per rank, handles exchanged over gloo, kernels on IPC-mapped peer memory.

    python -m torch.distributed.run --nnodes=1 --nproc-per-node W \\
        --master-addr 127.0.0.1 --master-port P tests/multirank_parity.py \\
        [--cases small,full,nvls] [--rounds 3]

Rank r runs on GPU ``LOCAL_RANK mod n_gpus``: on a 1-GPU box every rank shares
GPU 0 (CUDA IPC between processes on one device), on an N-GPU box the traffic
crosses NVLink.  Every case builds a cluster, runs a few rounds on deterministic
gradients and compares, BIT FOR BIT (tolerance only for the NVLS cases at
world > 2, where the switch's summation order is its own: the SGD cases hold the
switch's sum itself to 2e-6, the Adam cases 99.9 % of the elements to 2e-6 and all
of them to 5e-3 -- Adam amplifies a one-ulp change of a cancelling sum),

  * every hosted shard's var / m / v / beta powers / global_step with
    ``oracle.ps_oracle.CShard`` fed the same gradients (reference semantics:
    examples/mnist/mnist_replica.py:147-157 -- Adam on the PS, SURVEY appendix A),
  * every rank's pulled parameters, stripe by stripe, with the owners' oracle
    values (CRC32 of the bytes, exchanged over gloo).

Test infrastructure: launched by tests/test_gpu_multirank.py; also run by hand on
2/4/8 GPUs with the logs kept under profiles/.
"""
import argparse
import os
import sys
import time
import zlib

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

F = np.float32
MLP = [("global_step", ()), ("hid_w", (784, 100)), ("hid_b", (100,)), ("sm_w", (100, 10)),
       ("sm_b", (10,))]                                   # mnist_replica.py:121-134
NMF = [("W", (1_000_000, 200)), ("H", (200, 1_000))]      # matrix_factorization.py:21-28, scaled


def grad_np(lo, hi, seed):
    """Elements [lo, hi) of the deterministic gradient `seed` -- exact integer hash
    mapped to (-0.1, 0.1); torch on the GPU computes the same bits (grad_torch)."""
    idx = np.arange(lo, hi, dtype=np.int64)
    h = (idx * 2654435761 + seed * 40503 + 12345) & 0xFFFFFF
    return ((h.astype(F) / F(16777216.0) - F(0.5)) * F(0.2)).astype(F)


def grad_torch(n, seed, device):
    import torch
    idx = torch.arange(n, dtype=torch.int64, device=device)
    h = (idx * 2654435761 + seed * 40503 + 12345) & 0xFFFFFF
    return (h.to(torch.float32) / 16777216.0 - 0.5) * torch.tensor(0.2, dtype=torch.float32,
                                                                   device=device)


def seed_of(worker, rnd, task):
    return 1000 * worker + 10 * rnd + task


def bits(a):
    a = np.ascontiguousarray(a)
    return a.view(np.uint32) if a.dtype == np.float32 else a.view(np.uint16)


class Case(object):
    def __init__(self, name, variables, ps_tasks, placement=None, path="fused", wire="f32",
                 mode="sum", entry="round", stripes=None, ps_ranks=None, worker_ranks=None,
                 opt="adam", rtol=0.0):
        self.__dict__.update(locals())
        del self.__dict__["self"]


def build_cases(which, world):
    cases = []
    if "small" in which:
        for path in ("fused", "staged"):
            for wire in ("f32", "bf16"):
                for mode in ("sum", "mean", "async"):
                    cases.append(Case("mlp/%s/%s/%s/round" % (path, wire, mode), MLP, 1,
                                      path=path, wire=wire, mode=mode))
        cases.append(Case("mlp/fused/f32/sum/timer", MLP, 1, entry="timer"))
        cases.append(Case("mlp/fused/f32/async/graph", MLP, 1, mode="async", entry="graph"))
        cases.append(Case("mlp/staged/f32/sum/graph", MLP, 1, path="staged", entry="graph"))
        cases.append(Case("mlp/staged/f32/sum/round_host", MLP, 1, path="staged",
                          entry="round_host", stripes=max(4, world)))
        cases.append(Case("mlp/staged/bf16/mean/round_host", MLP, 1, path="staged", wire="bf16",
                          mode="mean", entry="round_host", stripes=max(4, world)))
        cases.append(Case("mlp/fused/f32/sum/sgd", MLP, 1, opt="sgd"))
        cases.append(Case("mlp/2ps/fused/f32/sum/stripes1", MLP, 2, stripes=1))
        if world >= 3:
            # PS shards on ranks that host no worker (tfrun's first-fit order: ps tasks
            # first, then workers -- script/tfrun:58-75, scheduler.py:252-275)
            cases.append(Case("mlp/dedicated-ps/fused/f32/sum", MLP, 1, ps_ranks=[0],
                              worker_ranks=list(range(1, world))))
            cases.append(Case("mlp/dedicated-ps/staged/bf16/async", MLP, 1, path="staged",
                              wire="bf16", mode="async", ps_ranks=[0],
                              worker_ranks=list(range(1, world))))
        if world >= 4:
            cases.append(Case("mlp/2ps-dedicated-striped/fused/f32/mean", MLP, 2, mode="mean",
                              ps_ranks=[[0, 1], [1, 0]], worker_ranks=list(range(2, world))))
    pl = {"W": 0, "H": 1}
    if "full" in which or "fullmin" in which:
        cases.append(Case("nmf/fused/f32/sum/round", NMF, 2, pl))        # the SCALE headline
        cases.append(Case("nmf/staged/f32/sum/round_host", NMF, 2, pl, path="staged",
                          entry="round_host", stripes=max(16, world)))   # the e2e configuration
    if "full" in which:
        cases.append(Case("nmf/fused/f32/sum/graph", NMF, 2, pl, entry="graph"))
        cases.append(Case("nmf/fused/bf16/async/round", NMF, 2, pl, wire="bf16", mode="async"))
    if "nvls" in which:
        tol = 0.0 if world <= 2 else 2e-6
        cases.append(Case("mlp/nvls/f32/sum/round", MLP, 1, path="nvls", rtol=tol))
        cases.append(Case("mlp/nvls/f32/mean/graph", MLP, 1, path="nvls", mode="mean",
                          entry="graph", rtol=tol))
        cases.append(Case("mlp/nvls/f32/sum/sgd", MLP, 1, path="nvls", opt="sgd", rtol=tol))
        cases.append(Case("mlp/nvls/f32/mean/sgd", MLP, 1, path="nvls", opt="sgd", mode="mean",
                          rtol=tol))
        if "full" in which or "nvlsfull" in which:
            cases.append(Case("nmf/nvls/f32/sum/round", NMF, 2, {"W": 0, "H": 1}, path="nvls",
                              rtol=tol))
    return cases


def run_case(case, rounds, rank, world, device, dist):
    import torch
    from oracle import ps_oracle as o
    from tfmesos_b200 import engine, psx

    modes = {"sum": (psx.MODE_SUM, o.SUM), "mean": (psx.MODE_SYNC_MEAN, o.SYNC_MEAN),
             "async": (psx.MODE_ASYNC_ORDERED, o.ASYNC_ORDERED)}
    pmode, omode = modes[case.mode]
    wire = psx.BF16 if case.wire == "bf16" else psx.F32
    if case.opt == "adam":
        optimizer, oopt = engine.AdamOptimizer(0.01), o.ADAM
    else:
        optimizer, oopt = engine.GradientDescentOptimizer(0.05), o.SGD
    cl = engine.TorchrunCluster(case.variables, case.ps_tasks, optimizer,
                                placement=case.placement, stripes=case.stripes, wire=wire,
                                device=device, path=case.path, ps_ranks=case.ps_ranks,
                                worker_ranks=case.worker_ranks)
    W = cl.n_workers
    dev = torch.device("cuda", device)
    wk, ws = cl.worker, cl.worker_stream
    tdt = torch.bfloat16 if wire == psx.BF16 else torch.float32

    # initial parameters: deterministic, non-zero, set by every owner on its shards
    refs = {}
    for key, ps in cl.servers.items():
        sp = ps.spec
        ref = o.CShard(sp.nelem, oopt, lr=optimizer.learning_rate)
        ref.var[:] = grad_np(sp.off, sp.off + sp.nelem, 777 + sp.task) * F(5.0)
        ps.shard.set_values(psx.VAR, ref.var)
        refs[key] = ref
    cl.barrier()

    def fill(rnd, host=False):
        if wk is None:
            return
        if host:
            # the last round_host's H2D copies read the pinned gradients
            # asynchronously (behind the other ranks' pushes); they are free
            # again once the worker stream has passed them
            ws.synchronize()
        for t in range(cl.layout.ps_tasks):
            n = wk.grad_flat[t].numel()
            if host:
                g = grad_torch(n, seed_of(wk.index, rnd, t), "cpu").to(tdt)
                cl.staging.grad[t].copy_(g)
            else:
                with torch.cuda.stream(ws):
                    wk.grad_flat[t].copy_(grad_torch(n, seed_of(wk.index, rnd, t), dev).to(tdt))

    graph = None
    if case.entry == "graph":
        fill(0)
        graph = cl.capture_round(pmode)
    if case.entry == "round_host" and wk is not None:
        cl.staging = engine.HostStaging(wk)
    timer = None
    if case.entry == "timer":
        class _T(object):
            def start(self, s): pass
            def stop(self, s): pass
        timer = _T()

    for rnd in range(1, rounds + 1):
        fill(rnd, host=case.entry == "round_host")
        if case.entry == "graph":
            with torch.cuda.stream(ws):
                graph.replay()
        elif case.entry == "round_host":
            if wk is not None:
                cl.round_host(pmode)
            else:
                for ps in cl.servers.values():       # PS-only rank: its applies of this round
                    ps.shard.apply_counted(pmode, 0, W, cl.ps_stream)
        else:
            cl.round(pmode, timer)
        # oracle for the shards hosted here (elementwise update: any sub-range is exact)
        for key, ps in cl.servers.items():
            sp = ps.spec
            slots = np.empty((W, sp.nelem), F)
            for w in range(W):
                g = grad_np(sp.off, sp.off + sp.nelem, seed_of(w, rnd, sp.task))
                if wire == psx.BF16:
                    g = o.bf16_to_f32(o.f32_to_bf16(g))
                slots[w] = g
            refs[key].round(slots, omode)
    cl.barrier()

    errors = []

    def same(got, want, what):
        if case.rtol == 0.0:
            if not np.array_equal(bits(got), bits(want)):
                bad = np.flatnonzero(bits(got) != bits(want))
                errors.append("%s: %d of %d elements differ (first %d: %r vs %r)"
                              % (what, bad.size, want.size, bad[0], got[bad[0]], want[bad[0]]))
        elif case.opt == "sgd":
            # var -= lr * g is linear in the reduced gradient: this checks the SWITCH's
            # W-way sum itself, to about one ulp of the gradient sum
            if not np.allclose(got, want, rtol=case.rtol, atol=case.rtol):
                d = np.abs(got - want)
                errors.append("%s: max abs diff %g (rtol %g)" % (what, float(d.max()), case.rtol))
        else:
            # Adam's step is ~alpha * sign(g) however small |g| is, so where the W-way
            # sum cancels to within ~1e-6 of zero a one-ulp reordering of the sum moves
            # the update by a visible fraction of lr (measured at W = 4: 1e-4 after 3
            # rounds on < 1e-4 of the elements).  Bar: 99.9 % of the elements within
            # 2e-6, every element within 5e-3.
            d = np.abs(got.astype(np.float64) - want)
            out = float(np.count_nonzero(d > case.rtol)) / max(1, d.size)
            if out > 1e-3 or float(d.max()) > 5e-3:
                errors.append("%s: %.2e of the elements beyond %g, max abs diff %g"
                              % (what, out, case.rtol, float(d.max())))

    crcs = {}
    for key, ps in cl.servers.items():
        ref = refs[key]
        same(ps.shard.get_values(psx.VAR), ref.var, "shard %r var" % (key,))
        if oopt == o.ADAM:
            same(ps.shard.get_values(psx.M), ref.m, "shard %r m" % (key,))
            same(ps.shard.get_values(psx.V), ref.v, "shard %r v" % (key,))
        st = ps.shard.state()
        want_step = rounds * (W if case.mode == "async" else 1)
        if st["global_step"] != want_step or ref.step != want_step:
            errors.append("shard %r global_step %d, oracle %d, expected %d"
                          % (key, st["global_step"], ref.step, want_step))
        if oopt == o.ADAM and (F(st["beta1_power"]) != ref.b1p or F(st["beta2_power"]) != ref.b2p):
            errors.append("shard %r beta powers %r/%r, oracle %r/%r"
                          % (key, st["beta1_power"], st["beta2_power"], ref.b1p, ref.b2p))
        want = o.f32_to_bf16(ref.var) if wire == psx.BF16 else ref.var
        crcs[key] = (zlib.crc32(np.ascontiguousarray(want).tobytes()), want)
    # every rank's pulled parameters, stripe by stripe, against the owners' oracle
    table = [None] * world
    dist.all_gather_object(table, {k: v[0] for k, v in crcs.items()})
    want_crc = {}
    for d in table:
        want_crc.update(d)
    if wk is not None:
        for sp in cl.topo.shards:
            src = cl.staging.param[sp.task] if case.entry == "round_host" else wk.param_flat[sp.task]
            got = src[sp.off:sp.off + sp.nelem]
            got = (got.view(torch.int16) if wire == psx.BF16 else got).cpu().numpy()
            if wire == psx.BF16:
                got = got.view(np.uint16)
            if case.rtol == 0.0:
                if zlib.crc32(np.ascontiguousarray(got).tobytes()) != want_crc[sp.key]:
                    if sp.key in crcs:
                        same(got, crcs[sp.key][1], "pulled params of shard %r" % (sp.key,))
                    else:
                        errors.append("pulled params of shard %r: CRC differs from the owner's "
                                      "oracle" % (sp.key,))
            elif sp.key in crcs:
                same(got, crcs[sp.key][1], "pulled params of shard %r" % (sp.key,))
    cl.close()
    return errors


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--cases", default="small")
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--only", default=None, help="substring filter on case names")
    args = ap.parse_args()
    import torch
    import torch.distributed as dist
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    n_gpus = torch.cuda.device_count()
    assert n_gpus >= 1, "multirank_parity needs a CUDA device: there is no CPU fallback"
    device = local % n_gpus
    torch.cuda.set_device(device)
    os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
    dist.init_process_group("gloo")
    which = set(args.cases.split(","))
    failed = 0
    for case in build_cases(which, world):
        if args.only and args.only not in case.name:
            continue
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
            print("CASE %-44s world=%d gpus=%d %s (%.1fs)"
                  % (case.name, world, min(world, n_gpus), "FAIL" if flag.item() else "ok",
                     time.time() - t0), flush=True)
        failed += int(flag.item() > 0)
        if errors and any(e.startswith("exception") for e in errors):
            break                                      # state after an exception is unknown
    dist.barrier()
    dist.destroy_process_group()
    if rank == 0:
        print("MULTIRANK PARITY: %s" % ("FAILED (%d cases)" % failed if failed else "all ok"),
              flush=True)
    sys.exit(1 if failed else 0)


if __name__ == "__main__":
    main()
