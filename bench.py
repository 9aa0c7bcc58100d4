#!/usr/bin/env python
"""bench.py -- PS push+pull GB/s and steps/sec of the B200 parameter-server path.

    python bench.py [--gpus N --steps K --warmup W]            # this repo's CUDA path
    python bench.py --impl reference [...]                      # the CPU-PS path

Workload (BASELINE.json configs[2], the one the GB/s metric is meaningful on):
the scaled matrix-factorization parameter set -- W (1e6 x 200) on ps:0 and
H (200 x 1e3) on ps:1 (placement of examples/matrix_factorization.py:21-28),
f32, Adam fused into the PS reduction -- one PS round per step: every worker
PUSHes its dense gradient, the PS reduces + applies, every worker PULLs the new
parameters.  Gradients are synthetic (the model's fwd/bwd is outside the named
path).  One process per GPU; rank r is worker r and hosts the shards pinned to
GPU r (each bucket striped over all N GPUs unless --stripes says otherwise).

    value  = n_workers * n_params * 8 B / t_step      ("push+pull GB/s", SURVEY 8d)
    e2e    = the same through TorchrunCluster.round_host(): gradients start in
             pinned HOST memory and parameters are read back to the host, both
             copies inside the timed region.
A second, small section times MNIST-replica training steps (mnist_replica.py's
MLP, fwd/bwd on the GPU by torch, Adam on the PS) and reports steps/sec.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

NMF_ROWS, NMF_COLS, NMF_RANK = 1_000_000, 1_000, 200
WORKLOADS = {
    # name: (variables, ps_tasks, placement)
    "nmf_scaled": ([("W", (NMF_ROWS, NMF_RANK)), ("H", (NMF_RANK, NMF_COLS))], 2,
                   {"W": 0, "H": 1}),
    "nmf_reference": ([("W", (1000, 200)), ("H", (200, 1000))], 2, {"W": 0, "H": 1}),
    "resnet50_bucket": ([("flat", (25_557_032,))], 1, None),
    "mnist_mlp": ([("global_step", ()), ("hid_w", (784, 100)), ("hid_b", (100,)),
                   ("sm_w", (100, 10)), ("sm_b", (10,))], 1, None),
    "mnist_softmax": ([("W", (784, 10)), ("b", (10,)), ("global_step", ())], 1, None),
    # the other reading of BASELINE config #3: the PARAMETER is 1e6 x 1e3 (4 GB f32)
    "embedding_1e6x1e3": ([("P", (1_000_000, 1_000))], 1, None),
}
MODES = {"sum": 1, "async": 0, "mean": 2}
DUMP_BYTES = 48 << 20       # --dump-outputs: all arrays together stay below 64 MB


def parse():
    p = argparse.ArgumentParser()
    p.add_argument("--gpus", type=int, default=1)
    p.add_argument("--steps", type=int, default=20)
    p.add_argument("--warmup", type=int, default=5)
    p.add_argument("--impl", default="b200", choices=["b200", "reference"])
    p.add_argument("--workload", default="nmf_scaled", choices=sorted(WORKLOADS))
    p.add_argument("--mode", default="sum", choices=sorted(MODES))
    p.add_argument("--path", default="auto",
                   choices=["auto", "staged", "fused", "unicast", "nvls"],
                   help="staged = push kernel + apply kernel + pull kernel; "
                        "fused (= unicast) = one PS-side gather/apply/scatter kernel over P2P "
                        "loads/stores (psx_round); nvls = the same round with the NVSwitch "
                        "reducing the gather (multimem.ld_reduce) and replicating the scatter "
                        "(multimem.st); auto = nvls from 4 GPUs when the box supports "
                        "multicast, else fused")
    p.add_argument("--ps-ranks", default=None,
                   help="ranks hosting the PS tasks, e.g. '0,1' (task t on rank t) or "
                        "'0+1,1+0' (task striped over ranks); default: every bucket striped "
                        "over all ranks")
    p.add_argument("--worker-ranks", default=None,
                   help="ranks running a worker, e.g. '2,3,4,5' (BASELINE config #3 as "
                        "written: --ps-ranks 0,1 --worker-ranks 2,3,4,5); default: all")
    p.add_argument("--e2e-stripes", type=int, default=None,
                   help="shards per bucket of the host-in/host-out round (pipelining grain; "
                        "default 16 on one GPU -- measured 90.4 vs 87.7 GB/s with 32, profiles/"
                        "r24, r29 -- and 32 from 2 GPUs, where every GPU hosts 1/N of them)")
    p.add_argument("--no-verify", action="store_true",
                   help="skip the oracle check of what was timed (\"verified\" key)")
    p.add_argument("--stripes", type=int, default=None,
                   help="GPUs each bucket is striped over (default: all)")
    p.add_argument("--wire", default="f32", choices=["f32", "bf16"],
                   help="element type of the workers' gradient/parameter tensors "
                        "(the PS master is always f32; bf16 = BASELINE config #4)")
    p.add_argument("--no-e2e", action="store_true")
    p.add_argument("--no-staged", action="store_true")
    p.add_argument("--no-mnist", action="store_true")
    p.add_argument("--no-tfrun", action="store_true",
                   help="skip the tfrun / one-process-per-task MNIST step timing (N = 1 only)")
    p.add_argument("--no-cpu-baseline", action="store_true")
    p.add_argument("--cpu-sample-elems", type=int, default=100_000_000,
                   help="CPU arms: parameters per step -- the SAME absolute sample at every "
                        "N, pushed / pulled by N workers")
    p.add_argument("--dump-outputs", metavar="DIR", default=None,
                   help="after the timed steps, write the parameters worker 0 pulled in the "
                        "last one as DIR/<variable>.npy (float32; a variable too large for "
                        "its share of %d MiB is sampled at fixed, seeded positions)"
                        % (DUMP_BYTES >> 20))
    args = p.parse_args()
    if args.dump_outputs and args.impl != "b200":
        p.error("--dump-outputs writes what the CUDA path computed: use it with --impl b200")
    return args


def n_params(workload):
    total = 0
    for _, shape in WORKLOADS[workload][0]:
        k = 1
        for d in shape:
            k *= d
        total += k
    return total


def bind_to_gpu_numa_node(index):
    """Run this rank on the cores next to its GPU so that the pinned staging
    buffers (first touch) and the copy-engine traffic stay on the GPU's socket."""
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(index)
        words = pynvml.nvmlDeviceGetCpuAffinity(h, (os.cpu_count() + 63) // 64)
        cpus = [64 * i + b for i, w in enumerate(words) for b in range(64) if (w >> b) & 1]
        if cpus:
            os.sched_setaffinity(0, cpus)
        return len(cpus)
    except Exception:
        return 0


# ------------------------------------------------------------------ clocks ----
class ClockSampler(object):
    """nvidia-smi clocks / throttle reasons DURING the timed region."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index=0):
        self.rows, self.proc, self.thread = [], None, None
        self.index = index

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                 "--format=csv,noheader,nounits", "-lms", "100"],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except OSError:
            self.proc = None
            return
        self.thread = threading.Thread(target=self._read)
        self.thread.daemon = True
        self.thread.start()

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(5)
        except subprocess.TimeoutExpired:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                sm.append(float(r[0]))
                mx.append(float(r[1]))
            except (ValueError, IndexError):
                continue
            for name, cell in zip(names, r[3:7]):
                if cell.lower().startswith("active"):
                    reasons.add(name)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None,
                "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons)}


class KernelTimer(object):
    """CUDA-event pairs around ONE kernel's launches, on its launching stream."""

    def __init__(self):
        self.pairs, self._cur = [], None

    def start(self, stream):
        import torch
        self._cur = torch.cuda.Event(enable_timing=True)
        self._cur.record(stream)

    def stop(self, stream):
        import torch
        e = torch.cuda.Event(enable_timing=True)
        e.record(stream)
        self.pairs.append((self._cur, e))

    def mean_ms(self):
        if not self.pairs:
            return None
        return sum(a.elapsed_time(b) for a, b in self.pairs) / len(self.pairs)


# --------------------------------------------------------------- CPU arms ----
def parse_ranks(text):
    if text is None:
        return None
    out = []
    for part in text.replace(":", ",").split(","):      # "0,1" or "0:1" (tools/gpu.sh splits on commas)
        rs = [int(x) for x in part.split("+")]
        out.append(rs if len(rs) > 1 else rs[0])
    return out


def n_workers_of(args, world):
    wr = parse_ranks(args.worker_ranks)
    return len(wr) if wr is not None else world


def cpu_ps(args, rounds=12, warmup=2):
    """The reference's CPU-PS path, best case (oracle/ps_oracle.c
    psx_oracle_cpu_ps_round: memcpy push, Eigen-style threaded apply on the PS
    host cores, memcpy pull) on a bounded sample of the workload: the SAME number
    of parameters at every N, pushed and pulled by as many workers as the CUDA arm
    has.  Persistent pinned thread pool with work stealing, every range
    first-touched by its owning thread.

    The pool has as many threads as the container can actually run: the CPUs in
    its affinity mask capped by its cgroup CPU quota.  The pool's GPU boxes show 128
    CPUs but give the container a 16-core CFS quota; with 128 threads the round time
    was bimodal (7-20 ms inside the quota, 40-100 ms once throttled until the next
    100 ms period -- profiles/r22-r29, explained by profiles/r30: `nr_throttled`
    climbs), with 16 threads it is 15.0 +- 0.1 ms.  Reported: the MEDIAN round,
    with every round time in `sample`; `cores` = the threads that ran."""
    from oracle import ps_oracle as o
    n_full = n_params(args.workload)
    W = max(1, n_workers_of(args, max(1, args.gpus)))
    n = min(n_full, max(1_000_000, args.cpu_sample_elems))
    base = o.CpuPsBaseline(n, W, o.ADAM, lr=0.01)
    mode = {"sum": o.SUM, "async": o.ASYNC_ORDERED, "mean": o.SYNC_MEAN}[args.mode]
    threads = 0
    for _ in range(warmup):
        threads = base.round(mode)
    times = []
    for _ in range(max(3, rounds)):
        t0 = time.perf_counter()
        threads = base.round(mode)
        times.append(time.perf_counter() - t0)
    in_order = ["%.1f" % (t * 1e3) for t in times]
    times.sort()
    dt = times[len(times) // 2]
    gbs = W * n * 8 / dt / 1e9
    quota = o.cpu_quota_cores()
    sample = ("%d of %d parameters (%.1f%%), %d worker(s), memcpy transport, MEDIAN of %d rounds "
              "(best %.1f ms; rounds in ms: %s); pool of %d pinned threads = CPUs usable by the "
              "container (%d in the affinity mask, CPU quota %s cores), work stealing, "
              "first-touch by owner"
              % (n, n_full, 100.0 * n / n_full, W, len(times), times[0] * 1e3,
                 " ".join(in_order), int(threads), len(os.sched_getaffinity(0)),
                 ("%.0f" % quota) if quota else "none"))
    return {"value": gbs, "unit": "GB/s", "cores": int(threads), "kind": "port",
            "sample": sample, "ms_per_step_on_sample": dt * 1e3,
            "cpu_quota_cores": quota, "host_cores_online": os.cpu_count()}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    steps, warmup = max(1, args.steps), max(1, args.warmup)
    cb = cpu_ps(args, rounds=max(10, steps), warmup=warmup)
    n_full = n_params(args.workload)
    line = {
        "impl": "reference",
        "metric": "ps_push_pull_GBps", "value": cb["value"], "unit": "GB/s",
        "n_gpus": args.gpus, "steps": steps, "warmup": warmup,
        "ms_per_step": cb["ms_per_step_on_sample"], "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": workload_config(args, max(1, args.gpus), n_full),
        "cpu_baseline": {k: cb[k] for k in ("value", "unit", "cores", "kind", "sample")},
        "e2e": {"value": cb["value"], "unit": "GB/s", "h2d_bytes_per_step": 0,
                "d2h_bytes_per_step": 0},
        "note": "CPU restatement of the TF-0.12 PS path (TensorFlow itself cannot run "
                "here); the timed step is the bounded sample named in cpu_baseline.sample",
    }
    print(json.dumps(line), flush=True)


def workload_config(args, world, n_full):
    return {"workload": "%s: PS round (push+reduce/apply+pull) over %d f32 parameters, Adam(lr=0.01)"
                        % (args.workload, n_full),
            "discipline": args.mode, "path": args.path, "wire": args.wire,
            "parallelism": ("%d workers (1/GPU), %d ps tasks, buckets striped over %s GPU(s)"
                            % (world, WORKLOADS[args.workload][1],
                               args.stripes if args.stripes else world))
                           if not (args.ps_ranks or args.worker_ranks) else
                           ("%d GPUs: ps tasks on ranks %s, workers on ranks %s"
                            % (world, args.ps_ranks or "all", args.worker_ranks or "all")),
            "l2": "per-step inputs (%.0f MB of gradients per worker) exceed the 126 MB L2"
                  % (n_full * 4 / 1e6) if n_full * 4 > 126e6 else "L2 flushed between steps"}


# ---------------------------------------------------------------- GPU arm ----
def mnist_section(torch, engine, psx, world, rank, dist, model="mlp", steps=100, warmup=10):
    """Full training steps on the reference's two MNIST models, synthetic
    [100,784] batches, forward/backward by torch on the worker GPU, one PS round
    per step with async-ordered applies (one global step per worker push):
      mlp      examples/mnist/mnist_replica.py:124-157  784-100-10, Adam(0.01)
      softmax  examples/mnist/mnist.py:44-55            784-10, SGD(0.005)
    Returns global steps/sec."""
    if model == "mlp":
        variables, ps_tasks, placement = WORKLOADS["mnist_mlp"]
        optimizer, names = engine.AdamOptimizer(0.01), ["hid_w", "hid_b", "sm_w", "sm_b"]
    else:
        variables, ps_tasks, placement = WORKLOADS["mnist_softmax"]
        optimizer, names = engine.GradientDescentOptimizer(0.005), ["W", "b"]
    cl = engine.TorchrunCluster(variables, ps_tasks, optimizer, placement=placement, stripes=1)
    g = torch.Generator(device="cuda").manual_seed(1234 + rank)
    if rank == 0 and model == "mlp":
        import numpy as np
        rng = np.random.default_rng(1)
        cl.set_variable("hid_w", np.clip(rng.standard_normal((784, 100)), -2, 2) / 28)
        cl.set_variable("sm_w", np.clip(rng.standard_normal((100, 10)), -2, 2) / 10)
    cl.barrier()
    x = torch.rand(100, 784, device="cuda", generator=g)
    y = torch.nn.functional.one_hot(torch.randint(0, 10, (100,), device="cuda", generator=g),
                                    10).float()
    wk = cl.worker
    ws = cl.worker_stream

    def fwd_bwd():
        x.uniform_(0.0, 1.0)                    # a fresh synthetic batch every step
        ps = [wk.params[k].detach().requires_grad_(True) for k in names]
        if model == "mlp":
            h = torch.relu(x @ ps[0] + ps[1])
            p = torch.softmax(h @ ps[2] + ps[3], 1)
            loss = -(y * torch.log(torch.clamp(p, 1e-10, 1.0))).sum()
        else:
            p = torch.softmax(x @ ps[0] + ps[1], 1)
            loss = -(y * torch.log(p)).sum()
        grads = torch.autograd.grad(loss, ps)
        for k, gr in zip(names, grads):
            wk.grads[k].copy_(gr)

    graph = None

    whole = None

    def step():
        if whole is not None:
            with torch.cuda.stream(ws):
                whole.replay()
            return
        with torch.cuda.stream(ws):
            if graph is not None:
                graph.replay()
            else:
                fwd_bwd()
        cl.round(psx.MODE_ASYNC_ORDERED)

    with torch.cuda.stream(ws):
        wk.pull(0, ws)
    for _ in range(warmup):
        step()
    cl.barrier()
    # the worker's compute is launch-bound (20-odd tiny kernels): capture it once
    # in a CUDA graph; the PS round stays ordinary launches (its sequence numbers
    # change every step)
    whole = None
    try:
        # the whole step -- forward/backward AND the PS round (signal/push, counted
        # stream waits, apply, pull) -- as ONE graph: a replay is a training step
        whole = cl.capture_round(psx.MODE_ASYNC_ORDERED, pre=fwd_bwd)
    except Exception as exc:
        sys.stderr.write("mnist: whole-step graph capture failed (%s)\n" % str(exc)[:300])
        whole = None
        try:
            torch.cuda.synchronize()
        except Exception:
            pass
    if whole is None:
        try:
            g_ = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g_, stream=ws):
                fwd_bwd()
            graph = g_
        except Exception as exc:                # keep measuring, eagerly
            sys.stderr.write("mnist: CUDA graph capture failed (%s), running eagerly\n" % exc)
            graph = None
    for _ in range(warmup):
        step()
    cl.barrier()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record(ws)
    for _ in range(steps):
        step()
    ev1.record(ws)
    cl.barrier()
    dt = ev0.elapsed_time(ev1) * 1e-3
    t = torch.tensor([dt], dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    n_par = n_params("mnist_mlp" if model == "mlp" else "mnist_softmax")
    out = {"global_steps_per_sec": steps * world / t.item(), "rounds": steps,
           "workers": world, "params": n_par,
           "model": ("784-100-10 MLP, batch 100, Adam 0.01, async-ordered" if model == "mlp"
                     else "784-10 softmax regression, batch 100, SGD 0.005, async-ordered"),
           "worker_compute": ("whole step (fwd/bwd + PS round) in one CUDA graph"
                              if whole is not None else
                              "CUDA graph" if graph is not None else "eager"),
           "push_pull_GBps": steps * world * n_par * 8 / t.item() / 1e9,
           "timing": "CUDA events on the worker stream over %d rounds, max over ranks" % steps}
    cl.close()
    return out


# ------------------------------------------------- synthetic data + verification
def synth_np(idx, seed):
    """Synthetic gradient element(s) `idx` (global bucket indices, int64) of stream
    `seed`: exact integer hash -> (-0.01, 0.01).  numpy on the host and torch on
    any GPU produce the same bits, so what a step consumed can be re-derived
    anywhere (verification needs no copy of the gradients)."""
    import numpy as np
    h = (idx.astype(np.int64) * 2654435761 + seed * 40503 + 12345) & 0xFFFFFF
    return ((h.astype(np.float32) / np.float32(16777216.0) - np.float32(0.5))
            * np.float32(0.02)).astype(np.float32)


def synth_torch(out, seed):
    """Fill the 1-D tensor `out` (any float dtype, CUDA or pinned host) with stream
    `seed`, chunk by chunk (the int64 index temp of a 2e8-element bucket is 1.6 GB)."""
    import torch
    dev = out.device if out.is_cuda else torch.device("cpu")
    scale = torch.tensor(0.02, dtype=torch.float32, device=dev)
    n, step = out.numel(), 1 << 26
    for lo in range(0, n, step):
        hi = min(n, lo + step)
        idx = torch.arange(lo, hi, dtype=torch.int64, device=dev)
        h = (idx * 2654435761 + seed * 40503 + 12345) & 0xFFFFFF
        out[lo:hi].copy_(((h.to(torch.float32) / 16777216.0 - 0.5) * scale).to(out.dtype))


def grad_seed(worker_index, task):
    return 100 + 16 * worker_index + task


def verify_cluster(cl, mode_name, wire_name, dist, host=False, samples=1_000_000):
    """Did the rounds that were just timed compute the right thing?  For every
    shard hosted here, a strided sample (>= `samples` elements, or the whole
    shard) of var / m / v plus global_step / beta powers is compared with the
    oracle (oracle.ps_oracle.CShard) replaying the SAME number of rounds on the
    same synthetic gradients; every worker's pulled parameters are compared with
    the owners' oracle values at the same positions.  Bit-exact for the unicast
    paths.  On the NVLS path the switch sums the W copies in its own order; Adam's
    step is ~alpha*sign(g) however small |g| is, so where the W-way sum cancels to
    within ~1e-6 of zero a one-ulp reordering moves the update by a visible
    fraction of lr (measured at W = 4 after 25 rounds: 1.8e-5 of the elements
    beyond 1e-5, max 1.4e-3).  Bar: at most 1e-4 of the elements beyond 1e-5, none
    beyond 0.05; the switch's sum itself is held to one ulp by the SGD cases of
    tests/multirank_parity.py.
    The oracle is the CHECKER here, outside every timed region."""
    import numpy as np
    import torch
    from oracle import ps_oracle as o
    from tfmesos_b200 import psx
    omode = {"sum": o.SUM, "async": o.ASYNC_ORDERED, "mean": o.SYNC_MEAN}[mode_name]
    rounds, W = cl.seq, cl.n_workers
    exact = not cl.nvls or W <= 2
    cl.barrier()
    checked = mism = 0
    max_diff = 0.0
    notes = []

    def compare(got, want):
        nonlocal checked, mism, max_diff
        checked += want.size
        if got.dtype != np.float32:                     # bf16 bit patterns
            mism += int(np.count_nonzero(got != want))
            return
        if exact:
            mism += int(np.count_nonzero(got.view(np.uint32) != want.view(np.uint32)))
        else:
            d = np.abs(got.astype(np.float64) - want)
            max_diff = max(max_diff, float(d.max()) if d.size else 0.0)
            mism += int(np.count_nonzero(d > 1e-5))

    mine = {}
    for key, ps in cl.servers.items():
        sp = ps.spec
        stride = max(1, sp.nelem // samples)
        idx = np.arange(0, sp.nelem, stride, dtype=np.int64)
        slots = np.empty((W, idx.size), np.float32)
        for w in range(W):
            g = synth_np(idx + sp.off, grad_seed(w, sp.task))
            if wire_name == "bf16":
                g = o.bf16_to_f32(o.f32_to_bf16(g))
            slots[w] = g
        ref = o.CShard(idx.size, o.ADAM, lr=0.01)
        for _ in range(rounds):
            ref.round(slots, omode)
        compare(ps.shard.get_values(psx.VAR)[idx], ref.var)
        compare(ps.shard.get_values(psx.M)[idx], ref.m)
        compare(ps.shard.get_values(psx.V)[idx], ref.v)
        st = ps.shard.state()
        want_step = rounds * (W if mode_name == "async" else 1)
        if st["global_step"] != want_step or ref.step != want_step:
            mism += 1
            notes.append("shard %r global_step %d, expected %d" % (key, st["global_step"], want_step))
        if np.float32(st["beta1_power"]) != ref.b1p or np.float32(st["beta2_power"]) != ref.b2p:
            mism += 1
            notes.append("shard %r beta powers differ" % (key,))
        mine[key] = (stride, o.f32_to_bf16(ref.var) if wire_name == "bf16" else ref.var)
    table = [None] * cl.world
    if cl.world > 1:
        dist.all_gather_object(table, mine)
    else:
        table = [mine]
    want = {}
    for d in table:
        want.update(d)
    if cl.worker is not None:
        for sp in cl.topo.shards:
            stride, ref_var = want[sp.key]
            src = cl.staging.param[sp.task] if host else cl.worker.param_flat[sp.task]
            got = src[sp.off:sp.off + sp.nelem][::stride]
            if wire_name == "bf16":
                got = got.contiguous().view(torch.int16).cpu().numpy().view(np.uint16)
            else:
                got = got.cpu().numpy()
            compare(got, ref_var)
    tot = torch.tensor([checked, mism], dtype=torch.float64)
    mx = torch.tensor([max_diff], dtype=torch.float64)
    if cl.world > 1:
        dist.all_reduce(tot)
        dist.all_reduce(mx, op=dist.ReduceOp.MAX)
    checked, mism = int(tot[0].item()), int(tot[1].item())
    ok = mism == 0 if exact else (mism <= 1e-4 * checked and mx.item() <= 0.05)
    out = {"ok": bool(ok), "rounds_replayed": rounds, "elements_checked": checked,
           "mismatches": mism,
           "bar": "bit-exact vs oracle (var, m, v, beta powers, global_step, pulled params)"
                  if exact else "NVLS (switch-order summation): <= 1e-4 of the elements beyond "
                                "1e-5 of the oracle, none beyond 0.05"}
    if not exact:
        out["max_abs_diff"] = mx.item()
    if notes:
        out["notes"] = notes[:4]
    return out


def dump_index(numel, n_vars):
    """Positions of a variable that --dump-outputs writes: all of them when the
    variable fits its share of DUMP_BYTES, else a sorted sample drawn with a
    fixed seed -- the same positions on every run and in every build."""
    import numpy as np
    cap = DUMP_BYTES // 4 // max(1, n_vars)
    if numel <= cap:
        return None
    return np.sort(np.random.default_rng(0).choice(numel, cap, replace=False))


def dump_outputs(worker, out_dir):
    """Write what the timed round handed `worker` in its last step: every
    variable's pulled parameters, as float32 <out_dir>/<name>.npy."""
    import numpy as np
    import torch
    os.makedirs(out_dir, exist_ok=True)
    for name, t in worker.params.items():
        flat = t.reshape(-1)
        idx = dump_index(flat.numel(), len(worker.params))
        if idx is not None:
            flat = flat[torch.from_numpy(idx).to(flat.device)]
        np.save(os.path.join(out_dir, name + ".npy"), flat.float().cpu().numpy())


def resolve_path(args, world, psx, local_rank):
    if args.path in ("staged", "nvls"):
        return args.path
    if args.path in ("fused", "unicast"):
        return "fused"
    symmetric = not (args.ps_ranks or args.worker_ranks)
    if world >= 4 and symmetric and args.wire == "f32" and args.mode != "async":
        try:
            if psx.nvls_supported(local_rank):
                return "nvls"
        except RuntimeError:
            pass
    return "fused"


def nvlink_peaks():
    try:
        return json.load(open(os.path.join(ROOT, "profiles", "nvlink_peaks.json")))
    except Exception:
        return {}


def run_b200(args):
    import torch
    import torch.distributed as dist
    from tfmesos_b200 import engine, psx

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device -- the product path has no CPU fallback")
    torch.cuda.set_device(local_rank)
    all_cpus = os.sched_getaffinity(0)
    bind_to_gpu_numa_node(local_rank)
    if world > 1:
        # plumbing only (handle exchange, barriers, max-over-ranks): gloo over
        # loopback -- nothing on the measured path uses a collective library
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("gloo")
    steps, warmup = max(1, args.steps), max(3, args.warmup)
    mode = MODES[args.mode]
    variables, ps_tasks, placement = WORKLOADS[args.workload]
    n_full = n_params(args.workload)
    path = resolve_path(args, world, psx, local_rank)
    ps_ranks, worker_ranks = parse_ranks(args.ps_ranks), parse_ranks(args.worker_ranks)

    wire = psx.BF16 if args.wire == "bf16" else psx.F32
    esz = 2 if args.wire == "bf16" else 4

    def make_cluster(which, stripes):
        cl_ = engine.TorchrunCluster(variables, ps_tasks, engine.AdamOptimizer(0.01),
                                     placement=placement, stripes=stripes, wire=wire,
                                     device=local_rank, path=which, ps_ranks=ps_ranks,
                                     worker_ranks=worker_ranks)
        if cl_.worker is not None:
            for t, g in enumerate(cl_.worker.grad_flat):
                synth_torch(g, grad_seed(cl_.worker.index, t))
        torch.cuda.synchronize()
        return cl_

    nvls_note = None
    try:
        cl = make_cluster(path, args.stripes)
    except engine.NvlsUnavailable as exc:
        if args.path == "nvls":
            raise
        # `auto` picked the switch path from the device attribute, but building the
        # multicast team failed (on every rank alike): run the unicast kernel instead.
        # Decided here, once, at set-up -- never per call.
        nvls_note = "NVLS set-up failed, unicast round used: %s" % str(exc)[:200]
        path = "fused"
        cl = make_cluster(path, args.stripes)
    W = cl.n_workers

    # L2 flush buffer for workloads smaller than L2
    flush = None
    if n_full * 4 <= 126e6:
        flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")

    def one_step(timer=None, host=False):
        if flush is not None:
            with torch.cuda.stream(cl.worker_stream):
                flush.zero_()
        if host:
            cl.round_host(mode)
        else:
            cl.round(mode, timer)

    def timed(n_steps, host=False, timer=None):
        cl.barrier()
        ev0 = torch.cuda.Event(enable_timing=True)
        ev1 = torch.cuda.Event(enable_timing=True)
        launches0 = psx.launch_count()
        # a PS-only rank has no worker stream activity: time its PS stream instead
        st = cl.worker_stream if cl.worker is not None else cl.ps_stream
        ev0.record(st)
        for _ in range(n_steps):
            one_step(timer, host)
        ev1.record(st)
        cl.barrier()
        ms = torch.tensor([ev0.elapsed_time(ev1)], dtype=torch.float64)
        launches = torch.tensor([psx.launch_count() - launches0], dtype=torch.float64)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
            dist.all_reduce(launches, op=dist.ReduceOp.SUM)
        return ms.item() / n_steps, int(launches.item())

    for _ in range(warmup):
        one_step()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    timer = KernelTimer()
    ms_step, launches = timed(steps, timer=timer)
    if args.dump_outputs and cl.worker is not None and cl.worker.index == 0:
        dump_outputs(cl.worker, args.dump_outputs)
    bytes_step = W * n_full * 2 * esz           # W * N * (s_g + s_p)
    value = bytes_step / (ms_step * 1e-3) / 1e9
    verified = None if args.no_verify else verify_cluster(cl, args.mode, args.wire, dist)

    # dominant kernel: the fused reduce+apply (or gather/apply/scatter) kernel
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    hbm_peak = float(peaks.get("hbm_gbs", 6650.0))
    peak_src = "measured (MEASURED_PEAKS.json)" if peaks else "fallback (B200_PROFILING.md)"
    # the kernel timer lives on the rank that hosts the largest shard; ranks without
    # one (worker-only) contribute nothing
    k_ms = timer.mean_ms() or 0.0
    shard_elems = ((cl.dominant.spec.nelem + 1023) // 1024) * 1024 if cl.dominant else 0
    if world > 1:
        # report the SLOWEST rank's dominant kernel (and its shard size)
        pair = torch.tensor([k_ms, float(shard_elems)], dtype=torch.float64)
        allp = [torch.zeros(2, dtype=torch.float64) for _ in range(world)]
        dist.all_gather(allp, pair)
        k_ms, shard_elems = max((p[0].item(), int(p[1].item())) for p in allp)
    if path == "nvls":
        per_elem = 24 + esz + esz              # var/m/v r+w, ONE reduced gradient in, ONE multicast store out
        kname = "k_round_mc<ADAM,%s> (multimem.ld_reduce + multimem.st)" % args.mode
    elif path == "fused":
        per_elem = 24 + esz * W + esz * W      # var/m/v r+w, W gradient reads, W param writes
        kname = "k_apply<ADAM,%s,SCATTER,PeerSrc<%s>>" % (args.mode, args.wire)
    else:
        per_elem = 24 + esz * W                # var/m/v r+w, W landing-slot reads
        kname = "k_apply<ADAM,%s,SlotSrc<%s>>" % (args.mode, args.wire)
    roofline = None
    if k_ms:
        # the timer brackets the launches over the largest shard only
        bytes_per_launch = per_elem * shard_elems
        achieved = bytes_per_launch / (k_ms * 1e-3) / 1e9
        traffic = nvl_measured = None
        try:
            tr = json.load(open(os.path.join(ROOT, "profiles", "roofline_traffic.json")))
            traffic = tr.get("%s/%s/n%d" % (args.workload, path, world))
            nvl_measured = tr.get("nvlink/%s" % path)
        except Exception:
            pass
        roofline = {"bound": "hbm", "kernel": kname, "achieved": achieved, "peak": hbm_peak,
                    "unit": "GB/s", "frac": achieved / hbm_peak, "traffic": traffic,
                    "peak_source": peak_src, "avg_launch_ms": k_ms,
                    "algorithmic_bytes_per_elem": per_elem,
                    "algorithmic_bytes_per_launch": bytes_per_launch,
                    "launches_timed": len(timer.pairs)}
        n_ps_gpus = len({s_.device for s_ in cl.topo.shards})
        if world > 1 and path in ("fused", "nvls") and n_ps_gpus > 1 or \
                (world > 1 and path == "fused" and (ps_ranks or worker_ranks)):
            # bound by this GPU's NVLink port, not by HBM.  Bytes per direction through
            # the port of the GPU that runs the kernel, while all stripes' kernels run:
            #   unicast: (W - own) remote gradient stripes in + the other owners'
            #            parameter stripes in (mirror image out): 2 (N-1) S for the
            #            symmetric layout, W S for a PS GPU that hosts no worker
            #   nvls:    N S gradient copies out + S multicast out, S reduced + N S
            #            parameters in: (N + 1) S
            S = shard_elems * esz
            if path == "nvls":
                nvl_bytes = (world + 1) * S
            elif ps_ranks or worker_ranks:
                nvl_bytes = W * S
            else:
                nvl_bytes = 2 * (world - 1) * S
            nvl = nvl_bytes / (k_ms * 1e-3) / 1e9
            pk = nvlink_peaks()
            duplex = pk.get("duplex_read_write_GBps")
            roofline.update({"bound": "nvlink", "achieved": nvl, "peak": 770.0,
                             "frac": nvl / 770.0,
                             "peak_source": "measured peer copy per direction "
                                            "(B200_PROFILING.md)",
                             "nvlink_bytes_per_direction_per_launch": nvl_bytes,
                             "frac_of_measured_duplex": (nvl / duplex) if duplex else None,
                             "measured_duplex_peak": duplex,
                             "measured_peaks_file": "profiles/nvlink_peaks.json" if pk else None,
                             "traffic": traffic,
                             "traffic_note": "NVLink bytes are algorithmic: ncu cannot attach "
                                             "to a multi-rank run here; nvlink_traffic_measured "
                                             "(when present) is ncu's nvlrx/nvltx count of this "
                                             "kernel in a one-process 2-GPU capture, as a ratio "
                                             "to the algorithmic bytes",
                             "nvlink_traffic_measured": nvl_measured,
                             "hbm_achieved": achieved, "hbm_frac": achieved / hbm_peak})
    resolved_stripes = len(cl.topo.shards_of(0))
    cl.close()

    ab = None
    if path == "nvls" and not args.no_staged:
        # A/B: the unicast one-kernel round on the same workload
        cl = make_cluster("fused", args.stripes)
        for _ in range(warmup):
            one_step()
        t3 = KernelTimer()
        ms_uni, l_uni = timed(max(3, steps // 2), timer=t3)
        v_uni = None if args.no_verify else verify_cluster(cl, args.mode, args.wire, dist)
        ab = {"path": "fused (unicast P2P loads/stores)", "value": bytes_step / (ms_uni * 1e-3) / 1e9,
              "unit": "GB/s", "ms_per_step": ms_uni, "kernel_avg_launch_ms": t3.mean_ms(),
              "verified": v_uni}
        cl.close()

    staged = None
    if path != "staged" and not args.no_staged:
        # the three-kernel path (push -> landing slot, reduce+apply, pull), the one
        # asynchronous / cross-process workers use; reported beside the headline
        cl = make_cluster("staged", args.stripes)
        for _ in range(warmup):
            one_step()
        t2 = KernelTimer()
        ms_staged, l_staged = timed(max(3, steps // 2), timer=t2)
        v_staged = None if args.no_verify else verify_cluster(cl, args.mode, args.wire, dist)
        per = 24 + esz * W
        staged = {"value": bytes_step / (ms_staged * 1e-3) / 1e9, "unit": "GB/s",
                  "ms_per_step": ms_staged, "gpu_launches": l_staged, "verified": v_staged}
        if t2.mean_ms():
            se = ((cl.dominant.spec.nelem + 1023) // 1024) * 1024
            staged["apply_kernel"] = {
                "kernel": "k_apply<ADAM,%s,SlotSrc<%s>>" % (args.mode, args.wire),
                "avg_launch_ms": t2.mean_ms(), "algorithmic_bytes_per_elem": per,
                "achieved": per * se / (t2.mean_ms() * 1e-3) / 1e9,
                "frac": per * se / (t2.mean_ms() * 1e-3) / 1e9 / hbm_peak}
        cl.close()

    e2e = None
    if not args.no_e2e:
        # same workload through the host-in / host-out public call; more, smaller
        # shards per bucket so H2D, the kernels and D2H pipeline across shards
        e2e_stripes = max(args.e2e_stripes or (16 if world == 1 else 32), world)
        cl = make_cluster("staged", e2e_stripes)
        if cl.worker is not None:
            cl.staging = engine.HostStaging(cl.worker)
            for t, g in enumerate(cl.staging.grad):
                synth_torch(g, grad_seed(cl.worker.index, t))

        def host_step():
            if cl.worker is not None:
                cl.round_host(mode)
            else:                                  # PS-only rank: its applies of this round
                cl.seq += 1
                for ps in cl.servers.values():
                    ps.shard.apply_counted(mode, 0, W, cl.ps_stream)

        _one = one_step
        one_step = lambda timer=None, host=False: host_step()  # noqa: E731
        for _ in range(2):
            one_step()
        ms_e2e, _ = timed(max(3, steps // 2), host=True)
        one_step = _one
        v_e2e = None if args.no_verify else verify_cluster(cl, args.mode, args.wire, dist,
                                                           host=True)
        hb = cl.staging.h2d_bytes() if cl.worker is not None else 0
        db = cl.staging.d2h_bytes() if cl.worker is not None else 0
        e2e = {"value": bytes_step / (ms_e2e * 1e-3) / 1e9, "unit": "GB/s",
               "ms_per_step": ms_e2e,
               "h2d_bytes_per_step": hb, "d2h_bytes_per_step": db,
               "stripes_per_bucket": e2e_stripes, "verified": v_e2e,
               "api": "tfmesos_b200.engine.TorchrunCluster.round_host (pinned host "
                      "gradients in, host parameters out, per rank; H2D / kernels / D2H "
                      "pipelined over the shards)"}
        cl.close()

    # clocks were sampled across all timed regions above (headline, staged, e2e)
    clocks = sampler.stop() if rank == 0 else None

    mnist = softmax = None
    if not args.no_mnist and not (ps_ranks or worker_ranks):
        mnist = mnist_section(torch, engine, psx, world, rank, dist, "mlp")
        softmax = mnist_section(torch, engine, psx, world, rank, dist, "softmax")

    # the LITERAL reference-API path next to the graph-captured one: tfrun + one OS
    # process per ps / worker task + examples/mnist/mnist_replica.py, request-free
    # async (tools/bench_tfrun.py).  1-GPU runs only: the tasks need the GPU to
    # themselves (this process is idle meanwhile), and it is a per-box latency figure.
    tfrun_api = None
    if rank == 0 and world == 1 and not args.no_mnist and not args.no_tfrun:
        try:
            sys.path.insert(0, os.path.join(ROOT, "tools"))
            import bench_tfrun
            torch.cuda.synchronize()
            torch.cuda.empty_cache()
            tfrun_api = {"command": "tfrun -w 1 -s 1 -- python examples/mnist/mnist_replica.py "
                                    "... --train_steps 1500 (one process per task, async Adam)"}
            for name, extra in (("as_the_reference_feeds_it(numpy batches, exact global_step)", []),
                                ("device_batches_lagged_step", ["--device_batches", "--lag_step"])):
                r = bench_tfrun.run(1, extra, 1500, timeout=90)
                tfrun_api[name] = ({"ms_per_step": r.get("ms_per_chief_step_median"),
                                    "steps_per_sec": (1e3 / r["ms_per_chief_step_median"]
                                                      if r.get("ms_per_chief_step_median") else None),
                                    "final_global_step": r.get("final_global_step")}
                                   if "error" not in r else {"error": r["error"][-200:]})
        except Exception as exc:                   # never lose the bench line over this
            tfrun_api = {"error": str(exc)[:200]}

    cpu = cpu_grpc = None
    if rank == 0 and not args.no_cpu_baseline:
        os.sched_setaffinity(0, all_cpus)          # the CPU arm gets every host core
        args.gpus = world
        cb = cpu_ps(args, rounds=10, warmup=2)
        cpu = {k: cb[k] for k in ("value", "unit", "cores", "kind", "sample")}
        if world == 1:
            try:
                # the same path over the transport the reference actually selects
                # (protocol='grpc'): loopback gRPC, one RPC per variable per direction
                from oracle import cpu_ps_grpc
                cpu_grpc = cpu_ps_grpc.time_round(min(n_full, 10_000_000), steps=3, warmup=1)
                cpu_grpc.update({"kind": "port", "transport": "python grpcio, loopback, raw "
                                 "bytes (TensorFlow's C++ gRPC core moves tensors a few times "
                                 "faster; the memcpy figure above is the upper bound for this "
                                 "path)"})
            except Exception as exc:
                cpu_grpc = {"unavailable": str(exc)[:200]}

    if rank == 0:
        cfg = workload_config(args, world, n_full)
        line = {
            "metric": "ps_push_pull_GBps", "value": value, "unit": "GB/s",
            "n_gpus": world, "steps": steps, "warmup": warmup, "ms_per_step": ms_step,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32" if args.wire == "f32" else "f32 master / bf16 wire",
            "data": "synthetic",
            "config": cfg,
            "path_resolved": path, "path_note": nvls_note, "n_workers": W, "stripes_per_bucket": resolved_stripes,
            "verified": verified["ok"] if verified else None,
            "verification": verified,
            "steps_per_sec": 1e3 / ms_step * (W if args.mode == "async" else 1),
            "gpu_launches": launches,
            "clocks": clocks,
            "roofline": roofline,
            "unicast_ab": ab,
            "staged_path": staged,
            "e2e": e2e,
            "cpu_baseline": cpu,
            "cpu_baseline_grpc": cpu_grpc,
            "mnist_replica": mnist,
            "mnist_softmax_sgd": softmax,
            "mnist_replica_via_tfrun": tfrun_api,
        }
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def main():
    args = parse()
    if args.impl == "reference":
        run_reference(args)
    else:
        run_b200(args)


if __name__ == "__main__":
    main()
