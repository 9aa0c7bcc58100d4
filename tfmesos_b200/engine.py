"""Host side of the PS data plane: the pieces of TensorFlow's between-graph
replication that the reference's examples use, re-expressed over libpsx.so.

    replica_device_setter      examples/mnist/mnist.py:43, mnist_replica.py:116
    GradientDescentOptimizer   mnist.py:55, matrix_factorization.py:39
    AdamOptimizer              mnist_replica.py:147
    MomentumOptimizer, AdagradOptimizer, RMSPropOptimizer
                               TF 0.12's tf.train classes of the same names
    ParameterServer            the process behind tf.train.Server for job 'ps'
                               (tfmesos/server.py:51-66, mnist_replica.py:93-95)
    Worker                     the session a worker opens on the PS devices
                               (mnist.py:65, mnist_replica.py:183)

Logical placement is the reference's: whole variables, round-robin over PS
tasks in creation order.  Physical layout is B200-first: all variables of one
PS task live in ONE flat f32 bucket in that GPU's HBM (one kernel per round,
not one RPC per variable), and a bucket may additionally be striped over
several GPUs to spread the NVLink ingress (SURVEY.md 7.3).
"""
import os
from collections import OrderedDict

from . import psx

ALIGN = 32          # variables start on 128-byte boundaries inside a bucket
STRIPE_ALIGN = 1024  # stripes start on 4 KiB boundaries


class GradientDescentOptimizer(object):
    """tf.train.GradientDescentOptimizer(learning_rate) (mnist.py:55).

    Every optimizer class carries ``opt`` (the PSX_OPT_* id) and ``hyper``, the
    four floats the shard header holds (include/psx.h lists their meaning)."""
    opt = psx.OPT_SGD

    def __init__(self, learning_rate):
        self.learning_rate = float(learning_rate)
        # the unused slots keep Adam's defaults: the header's stored powers, and so
        # the checkpoint metadata, stay what they have always been for SGD
        self.hyper = (self.learning_rate, 0.9, 0.999, 1e-8)


class AdamOptimizer(object):
    """tf.train.AdamOptimizer(learning_rate) with TF's defaults (mnist_replica.py:147)."""
    opt = psx.OPT_ADAM

    def __init__(self, learning_rate=0.001, beta1=0.9, beta2=0.999, epsilon=1e-8):
        self.learning_rate = float(learning_rate)
        self.beta1, self.beta2, self.epsilon = float(beta1), float(beta2), float(epsilon)
        self.hyper = (self.learning_rate, self.beta1, self.beta2, self.epsilon)


class MomentumOptimizer(object):
    """tf.train.MomentumOptimizer(learning_rate, momentum) (use_nesterov=False):
    accum = accum * momentum + grad; var -= accum * lr.  accum starts at 0."""
    opt = psx.OPT_MOMENTUM

    def __init__(self, learning_rate, momentum):
        self.learning_rate, self.momentum = float(learning_rate), float(momentum)
        self.hyper = (self.learning_rate, self.momentum, 0.0, 0.0)


class AdagradOptimizer(object):
    """tf.train.AdagradOptimizer(learning_rate, initial_accumulator_value=0.1):
    accum += grad^2; var -= grad * lr / sqrt(accum).  accum starts at
    initial_accumulator_value, which must be positive."""
    opt = psx.OPT_ADAGRAD

    def __init__(self, learning_rate, initial_accumulator_value=0.1):
        if not initial_accumulator_value > 0.0:
            raise ValueError("initial_accumulator_value must be positive: %r"
                             % (initial_accumulator_value,))
        self.learning_rate = float(learning_rate)
        self.initial_accumulator_value = float(initial_accumulator_value)
        self.hyper = (self.learning_rate, self.initial_accumulator_value, 0.0, 0.0)


class RMSPropOptimizer(object):
    """tf.train.RMSPropOptimizer(learning_rate, decay=0.9, momentum=0.0,
    epsilon=1e-10) (centered=False): ms += (grad^2 - ms) * (1 - decay);
    mom = mom * momentum + grad * lr / sqrt(ms + epsilon); var -= mom.
    ms starts at 1 (TF's ``rms`` slot), mom at 0."""
    opt = psx.OPT_RMSPROP

    def __init__(self, learning_rate, decay=0.9, momentum=0.0, epsilon=1e-10):
        self.learning_rate = float(learning_rate)
        self.decay, self.momentum, self.epsilon = float(decay), float(momentum), float(epsilon)
        self.hyper = (self.learning_rate, self.decay, self.momentum, self.epsilon)


def replica_device_setter(ps_tasks=0, cluster=None):
    """Returns ``place(name) -> ps task index``: round-robin per variable in
    creation order, starting at task 0 (tf.train.replica_device_setter as called
    at mnist.py:43 with ps_tasks= and at mnist_replica.py:116 with cluster=).
    Optimizer slots are colocated with their variable and never call this."""
    if cluster is not None:
        ps_tasks = len(cluster.get("ps", []))
    state = {"next": 0}

    def place(name):
        if ps_tasks <= 0:
            return None
        task = state["next"] % ps_tasks
        state["next"] += 1
        return task

    return place


def _round_up(x, a):
    return (x + a - 1) // a * a


class VariableLayout(object):
    """Which PS task owns each variable and where it sits in that task's bucket."""

    def __init__(self, variables, ps_tasks, placement=None):
        """variables: [(name, shape)] in creation order; placement: optional
        {name: task} for explicit tf.device pinning (matrix_factorization.py:21-28)."""
        self.ps_tasks = int(ps_tasks)
        self.entries = OrderedDict()
        self.bucket_nelem = [0] * self.ps_tasks
        place = replica_device_setter(ps_tasks=self.ps_tasks)
        for name, shape in variables:
            numel = 1
            for d in shape:
                numel *= int(d)
            if placement is not None and name in placement:
                task = placement[name]
            else:
                task = place(name)
            off = _round_up(self.bucket_nelem[task], ALIGN)
            self.entries[name] = (task, off, tuple(int(d) for d in shape), numel)
            self.bucket_nelem[task] = off + numel

    def placement(self):
        return OrderedDict((n, e[0]) for n, e in self.entries.items())

    def names_of(self, task):
        return [n for n, e in self.entries.items() if e[0] == task]


def stripe_ranges(nelem, stripes):
    """Split [0, nelem) into <= `stripes` contiguous ranges on 4 KiB boundaries."""
    stripes = max(1, int(stripes))
    chunk = _round_up(_round_up(nelem, stripes) // stripes, STRIPE_ALIGN)
    out = []
    lo = 0
    while lo < nelem:
        hi = min(nelem, lo + chunk)
        out.append((lo, hi - lo))
        lo = hi
    return out


class ShardSpec(object):
    def __init__(self, task, stripe, device, off, nelem):
        self.task, self.stripe, self.device = task, stripe, device
        self.off, self.nelem = off, nelem
        self.key = (task, stripe)

    def __repr__(self):
        return "ShardSpec(ps:%d/%d gpu%d [%d,+%d))" % (self.task, self.stripe, self.device,
                                                       self.off, self.nelem)


class Topology(object):
    """Every shard of every PS task and the GPU it is pinned to.  Deterministic,
    so all processes build the same object from the same arguments."""

    def __init__(self, layout, ps_devices, worker_devices):
        """ps_devices: per PS task, a device ordinal or a list of them (stripes);
        worker_devices: device ordinal per worker index."""
        self.layout = layout
        self.worker_devices = list(worker_devices)
        self.shards = []
        for task in range(layout.ps_tasks):
            devs = ps_devices[task]
            if isinstance(devs, int):
                devs = [devs]
            n = max(1, layout.bucket_nelem[task])
            for j, (off, cnt) in enumerate(stripe_ranges(n, len(devs))):
                self.shards.append(ShardSpec(task, j, devs[j], off, cnt))

    @property
    def n_workers(self):
        return len(self.worker_devices)

    def shards_on(self, device):
        return [s for s in self.shards if s.device == device]

    def shards_of(self, task):
        return [s for s in self.shards if s.task == task]


class ParameterServer(object):
    """One shard of one PS task, resident on one GPU."""

    def __init__(self, spec, optimizer, n_workers, wire=psx.F32, landing_slots=True,
                 device=None):
        """device: physical CUDA ordinal when it differs from the topology's logical
        one (several ranks sharing a GPU; CUDA_VISIBLE_DEVICES remapping)."""
        self.spec = spec
        self.n_workers = int(n_workers)
        self.device = spec.device if device is None else int(device)
        self.shard = psx.Shard(self.device, spec.nelem, optimizer.opt, *optimizer.hyper,
                               n_slots=self.n_workers if landing_slots else 0, wire=wire)

    def handle(self):
        return self.shard.export()

    def apply(self, mode, wait_seq=0, stream=None, first_slot=0, count=None):
        self.shard.apply(mode, first_slot, self.n_workers if count is None else count,
                         wait_seq, stream)

    def round(self, mode, wait_seq=0, stream=None, first_slot=0, count=None):
        self.shard.round(mode, first_slot, self.n_workers if count is None else count,
                         wait_seq, stream)

    def close(self):
        self.shard.destroy()


class Worker(object):
    """A worker's view of the whole parameter set: one flat gradient and one
    flat parameter tensor per PS task in ITS OWN HBM (what TF keeps as the
    worker-side copies it _Recv'd / will _Send), with per-variable views."""

    def __init__(self, index, topology, handles, exportable=False, wire=psx.F32, device=None,
                 arena=None):
        """handles: {(task, stripe): shard handle bytes}.  wire: element type of
        this worker's gradient / parameter tensors (f32, or bf16 for BASELINE
        config #4 -- the PS keeps f32 master copies either way).  device: physical
        CUDA ordinal if it differs from the topology's logical one.  arena: an
        object with ``carve(nbytes) -> (ptr, tensor_factory)`` that provides the
        staging memory instead of psx.Buffer (the NVLS multicast arena)."""
        import torch
        self.index = int(index)
        self.wire = wire
        dtype = torch.bfloat16 if wire == psx.BF16 else torch.float32
        esize = 2 if wire == psx.BF16 else 4
        self.topo = topology
        self.logical_device = topology.worker_devices[self.index]
        self.device = self.logical_device if device is None else int(device)
        self.layout = topology.layout
        dev = torch.device("cuda", self.device)
        self.buffers = []
        self.arena_offsets = []         # per task: (grad byte offset, param byte offset)
        self.grad_flat, self.param_flat = [], []
        for task in range(self.layout.ps_tasks):
            shards = topology.shards_of(task)
            n = _round_up(sum(s.nelem for s in shards), STRIPE_ALIGN)
            if arena is not None:
                goff, g = arena.carve(n * esize, dtype)
                poff, p = arena.carve(n * esize, dtype)
                self.arena_offsets.append((goff, poff))
                self.grad_flat.append(g)
                self.param_flat.append(p)
            elif exportable:    # psx_round needs IPC-exportable staging
                g, p = psx.Buffer(self.device, n * esize), psx.Buffer(self.device, n * esize)
                self.buffers.append((g, p))
                self.grad_flat.append(g.tensor(dtype))
                self.param_flat.append(p.tensor(dtype))
            else:
                self.grad_flat.append(torch.zeros(n, dtype=dtype, device=dev))
                self.param_flat.append(torch.zeros(n, dtype=dtype, device=dev))
        self.clients = OrderedDict()
        for s in topology.shards:
            self.clients[s.key] = psx.Client(handles[s.key], self.device, self.index)
        # Walk the shards starting with the ones on this worker's own GPU, then
        # GPU+1, GPU+2, ... : at any moment every GPU is the target of exactly one
        # worker (a permutation), instead of all workers converging on GPU 0 first
        # (incast: measured 8 ms vs ~3 ms per staged round at N=8, profiles/r08).
        ngpu = max([s.device for s in topology.shards] + list(topology.worker_devices)) + 1
        self.order = sorted(topology.shards,
                            key=lambda s: ((s.device - self.logical_device) % ngpu, s.task,
                                           s.stripe))
        self.params, self.grads = OrderedDict(), OrderedDict()
        for name, (task, off, shape, numel) in self.layout.entries.items():
            self.params[name] = self.param_flat[task][off:off + numel].view(shape)
            self.grads[name] = self.grad_flat[task][off:off + numel].view(shape)

    def client_handles(self):
        return {k: c.export() for k, c in self.clients.items()}

    def buffer_handles(self):
        return [(g.export(), p.export()) for g, p in self.buffers]

    def push(self, seq=0, stream=None):
        """PUSH every bucket stripe into this worker's slot on its PS GPU."""
        for s in self.order:
            g = self.grad_flat[s.task]
            self.clients[s.key].push(g.data_ptr() + s.off * g.element_size(), s.nelem, 0,
                                     self.wire, seq, stream)

    def pull(self, wait_seq=0, stream=None):
        """PULL every bucket stripe from its PS GPU into the flat parameters."""
        for s in self.order:
            p = self.param_flat[s.task]
            self.clients[s.key].pull(p.data_ptr() + s.off * p.element_size(), s.nelem, 0,
                                     self.wire, wait_seq, stream)

    def signal(self, seq, stream=None):
        for c in self.clients.values():
            c.signal(seq, stream)

    def wait_applied(self, seq, stream=None):
        for c in self.clients.values():
            c.wait_applied(seq, stream)

    def close(self):
        for c in self.clients.values():
            c.close()
        self.clients.clear()
        self.params.clear()
        self.grads.clear()
        self.grad_flat, self.param_flat = [], []
        for g, p in self.buffers:
            g.destroy()
            p.destroy()
        self.buffers = []


class LocalCluster(object):
    """All PS shards and all workers in THIS process (one or several GPUs):
    the in-graph shape of examples/mnist/mnist.py, and what the tests and the
    single-GPU bench use.  Multi-process deployments build the same objects per
    process and exchange the handle blobs over the rendez-vous socket."""

    def __init__(self, variables, ps_tasks, n_workers, optimizer, ps_devices=None,
                 worker_devices=None, placement=None, wire=psx.F32, fused=False):
        self.layout = VariableLayout(variables, ps_tasks, placement)
        if ps_devices is None:
            ps_devices = [0] * ps_tasks
        if worker_devices is None:
            worker_devices = [0] * n_workers
        self.topo = Topology(self.layout, ps_devices, worker_devices)
        self.servers = OrderedDict()
        for spec in self.topo.shards:
            self.servers[spec.key] = ParameterServer(spec, optimizer, n_workers, wire,
                                                     landing_slots=not fused)
        handles = {k: ps.handle() for k, ps in self.servers.items()}
        self.workers = [Worker(i, self.topo, handles, exportable=fused, wire=wire)
                        for i in range(n_workers)]
        for w in self.workers:
            for key, h in w.client_handles().items():
                self.servers[key].shard.register_client(w.index, h)
        if fused:
            for w in self.workers:
                for spec in self.topo.shards:
                    g, p = w.buffers[spec.task]
                    self.servers[spec.key].shard.round_bind(w.index, g.export(), p.export(),
                                                            spec.off)
        self.fused = fused
        self.seq = 0

    # -- whole-variable access on the PS (init_op / Variable.eval()) ---------
    def set_variable(self, name, value):
        import numpy as np
        task, off, shape, numel = self.layout.entries[name]
        flat = np.ascontiguousarray(value, dtype=np.float32).reshape(-1)
        assert flat.size == numel, (name, flat.size, numel)
        for spec in self.topo.shards_of(task):
            lo, hi = max(off, spec.off), min(off + numel, spec.off + spec.nelem)
            if lo < hi:
                self.servers[spec.key].shard.set_values(psx.VAR, flat[lo - off:hi - off],
                                                        lo - spec.off)

    def get_variable(self, name, which=psx.VAR):
        import numpy as np
        task, off, shape, numel = self.layout.entries[name]
        out = np.empty(numel, np.float32)
        for spec in self.topo.shards_of(task):
            lo, hi = max(off, spec.off), min(off + numel, spec.off + spec.nelem)
            if lo < hi:
                out[lo - off:hi - off] = self.servers[spec.key].shard.get_values(
                    which, lo - spec.off, hi - lo)
        return out.reshape(shape)

    def global_step(self):
        return next(iter(self.servers.values())).shard.state()["global_step"]

    # -- one PS round over all workers' gradients ----------------------------
    def round(self, mode, stream=None):
        """push (all workers) -> apply (all shards) -> pull (all workers)."""
        self.seq += 1
        if self.fused:
            for w in self.workers:
                w.signal(self.seq, stream)
            for ps in self.servers.values():
                ps.round(mode, self.seq, stream)
            for w in self.workers:
                w.wait_applied(self.seq, stream)
        else:
            for w in self.workers:
                w.push(self.seq, stream)
            for ps in self.servers.values():
                ps.apply(mode, self.seq, stream)
            for w in self.workers:
                w.pull(self.seq, stream)

    def close(self):
        for w in self.workers:
            w.close()
        for ps in self.servers.values():
            ps.close()
        self.servers.clear()
        self.workers = []


class HostStaging(object):
    """Pinned host mirrors of a worker's flat gradient / parameter tensors: the
    reference's worker keeps these in host memory (its PS path is CPU<->CPU over
    gRPC); with them the public round is host-in / host-out."""

    def __init__(self, worker):
        import torch
        self.grad = [torch.empty(t.numel(), dtype=t.dtype).pin_memory()
                     for t in worker.grad_flat]
        self.param = [torch.empty(t.numel(), dtype=t.dtype).pin_memory()
                      for t in worker.param_flat]

    def h2d_bytes(self):
        return sum(t.numel() * t.element_size() for t in self.grad)

    def d2h_bytes(self):
        return sum(t.numel() * t.element_size() for t in self.param)


def merge_across_ranks(mine):
    """all_gather a dict from every rank and merge them (handle exchange)."""
    import torch.distributed as dist
    if not dist.is_initialized() or dist.get_world_size() == 1:
        return dict(mine)
    out = [None] * dist.get_world_size()
    dist.all_gather_object(out, mine)
    merged = {}
    for d in out:
        merged.update(d)
    return merged


def torchrun_topology(layout, world, stripes=None, ps_ranks=None, worker_ranks=None):
    """Default: stripe j of PS task t is pinned to GPU (t + j) mod world and worker r
    runs on GPU r.  ``ps_ranks`` (one rank or list of ranks per PS task) and
    ``worker_ranks`` place them explicitly -- e.g. BASELINE config #3 as written,
    2 ps + 4 workers: ps_ranks=[0, 1], worker_ranks=[2, 3, 4, 5] (the first-fit
    order of tfmesos/scheduler.py:252-275: ps tasks first, then workers).
    Same arguments -> same topology on every rank."""
    if ps_ranks is None:
        stripes = world if stripes is None else max(1, int(stripes))
        ps_ranks = [[(t + j) % world for j in range(stripes)] for t in range(layout.ps_tasks)]
    else:
        ps_ranks = [[r] if isinstance(r, int) else list(r) for r in ps_ranks]
        if stripes is not None and len(ps_ranks) == layout.ps_tasks:
            # more stripes than listed ranks: cycle over them (pipelining granularity)
            ps_ranks = [[rs[j % len(rs)] for j in range(max(len(rs), int(stripes)))]
                        for rs in ps_ranks]
        assert len(ps_ranks) == layout.ps_tasks, "one rank (list) per PS task"
    if worker_ranks is None:
        worker_ranks = list(range(world))
    return Topology(layout, ps_ranks, list(worker_ranks))


class NvlsUnavailable(RuntimeError):
    """The NVSwitch multicast set-up failed on some rank; raised on EVERY rank, at
    cluster construction (the path is chosen at init, never per call)."""


class McArena(object):
    """This rank's member of one NVSwitch multicast object shared by all worker
    ranks (psx_mcx_*): a VMM allocation in this GPU's HBM that is mapped twice --
    at a unicast address (ordinary loads / stores: the torch views below) and,
    together with every other member's allocation, at ONE multicast address on
    which the switch executes multimem.ld_reduce (sum over all members) and
    multimem.st (store to all members).  The multicast object's POSIX fd goes from
    rank 0 to the other processes over an AF_UNIX socket (SCM_RIGHTS); CUDA-IPC
    blobs cannot carry it."""

    def __init__(self, device, nbytes, rank, world, broadcast):
        """broadcast(obj_or_None) -> obj: rank 0's object on every rank."""
        import socket
        self.device, self.rank, self.world = int(device), int(rank), int(world)
        self.cursor = 0
        fd = -1
        self.mcx = None
        if rank == 0:
            try:
                self.mcx = psx.McMember.create(device, world, nbytes)
            except RuntimeError:
                if world > 1:
                    broadcast(None)        # the others must not wait for a socket name
                raise
            fd = self.mcx.fd
        if world > 1:
            if rank == 0:
                name = "\0psx-mc-%d-%d" % (os.getpid(), id(self) & 0xFFFFFF)
                srv = socket.socket(socket.AF_UNIX, socket.SOCK_STREAM)
                srv.bind(name)
                srv.listen(world)
                srv.settimeout(120)
                broadcast(name)
                for _ in range(world - 1):
                    conn, _ = srv.accept()
                    socket.send_fds(conn, [b"mc"], [fd])
                    conn.recv(1)            # the peer has imported: its copy of the fd is live
                    conn.close()
                srv.close()
            else:
                name = broadcast(None)
                if name is None:
                    raise RuntimeError("rank 0 could not create the multicast object")
                c = socket.socket(socket.AF_UNIX, socket.SOCK_STREAM)
                c.settimeout(120)
                c.connect(name)
                _, fds, _, _ = socket.recv_fds(c, 16, 1)
                self.mcx = psx.McMember.import_fd(device, world, nbytes, fds[0])
                os.close(fds[0])
                c.send(b"k")
                c.close()
        self.mcx.add_device()

    def bind(self):
        """After EVERY member has added its device (barrier in between)."""
        self.uc, self.mc, self.size = self.mcx.bind()

    def carve(self, nbytes, dtype):
        import torch
        nbytes = _round_up(int(nbytes), 4096)
        off = self.cursor
        assert off + nbytes <= self.size, "multicast arena exhausted"
        self.cursor += nbytes
        esz = torch.empty(0, dtype=dtype).element_size()
        return off, psx.device_tensor(self.uc + off, nbytes // esz, dtype, self.device, self)

    def destroy(self):
        if self.mcx is not None:
            self.mcx.destroy()
            self.mcx = None


class TorchrunCluster(object):
    """One process per GPU (launched by torchrun / tfrun).  By default rank r is
    worker r on GPU r and also hosts the PS shards pinned to GPU r; ``ps_ranks`` /
    ``worker_ranks`` give other shapes (PS shards on GPUs that host no worker,
    idle ranks).  Handle blobs are exchanged once with all_gather_object --
    torch.distributed is plumbing only; nothing on the push/apply/pull path
    touches NCCL.

    path: "staged" (push kernel -> landing slot, reduce+apply kernel, pull kernel),
          "fused"  (one PS-side kernel gathers over P2P loads, applies, scatters
                    with P2P stores -- psx_round),
          "nvls"   (the same kernel with the gather done by the switch --
                    multimem.ld_reduce -- and the scatter by multimem.st).
    device: physical CUDA ordinal of this rank (default: its rank); ranks may share
    a GPU (tests on a 1-GPU box)."""

    def __init__(self, variables, ps_tasks, optimizer, placement=None, stripes=None,
                 fused=False, wire=psx.F32, device=None, ps_ranks=None, worker_ranks=None,
                 path=None):
        import torch
        import torch.distributed as dist
        self.rank = dist.get_rank() if dist.is_initialized() else 0
        self.world = dist.get_world_size() if dist.is_initialized() else 1
        self.device = self.rank if device is None else device
        if path is None:
            path = "fused" if fused else "staged"
        assert path in ("staged", "fused", "nvls"), path
        self.path = path
        self.nvls = path == "nvls"
        self.fused = fused = path in ("fused", "nvls")
        psx.init(self.device)
        self.layout = VariableLayout(variables, ps_tasks, placement)
        # more stripes than GPUs gives several independent shards per GPU (the
        # pipelining granularity of round_host)
        self.topo = torchrun_topology(self.layout, self.world, stripes, ps_ranks, worker_ranks)
        self.worker_ranks = list(self.topo.worker_devices)
        self.n_workers = len(self.worker_ranks)
        self.worker_index = (self.worker_ranks.index(self.rank)
                             if self.rank in self.worker_ranks else None)
        self.servers = OrderedDict()
        for spec in self.topo.shards_on(self.rank):
            self.servers[spec.key] = ParameterServer(spec, optimizer, self.n_workers, wire,
                                                     landing_slots=not fused,
                                                     device=self.device)
        handles = self._merge({k: ps.handle() for k, ps in self.servers.items()})
        self.arena = None
        if self.nvls:
            if self.worker_ranks != list(range(self.world)) or wire != psx.F32:
                raise RuntimeError("the NVLS round needs every rank to be a worker (all "
                                   "members contribute to multimem.ld_reduce) and an f32 wire")
            esize = 4
            need = sum(2 * _round_up(_round_up(sum(s.nelem for s in self.topo.shards_of(t)),
                                               STRIPE_ALIGN) * esize, 4096)
                       for t in range(self.layout.ps_tasks))
            # every stage is agreed on by all ranks before the next one starts: a rank
            # that fails must not leave the others waiting in a barrier / a bind
            try:
                self.arena = McArena(self.device, need, self.rank, self.world, self._bcast)
                err = None
            except (RuntimeError, OSError) as exc:
                err = "rank %d: %s" % (self.rank, str(exc)[:300])
            self._agree(err)
            self.barrier()                 # every member added its device ...
            try:
                self.arena.bind()          # ... before anyone binds memory
                err = None
            except RuntimeError as exc:
                err = "rank %d: %s" % (self.rank, str(exc)[:300])
            self._agree(err)
            self.barrier()
        self.worker = None
        self.mailbox = None
        if self.worker_index is not None:
            self.worker = Worker(self.worker_index, self.topo, handles,
                                 exportable=fused and not self.nvls, wire=wire,
                                 device=self.device, arena=self.arena)
        clients = self._merge({(k, self.worker_index): h
                               for k, h in (self.worker.client_handles().items()
                                            if self.worker else [])})
        for (key, widx), h in clients.items():
            if key in self.servers:
                self.servers[key].shard.register_client(widx, h)
        # counter rendez-vous: one mailbox per worker, bumped by every shard's apply
        if self.worker is not None:
            self.mailbox = psx.Mailbox(self.device)
        boxes = self._merge({self.worker_index: self.mailbox.export()}
                            if self.worker else {})
        for ps in self.servers.values():
            for widx, h in boxes.items():
                ps.shard.register_mailbox(widx, h)
        self.n_shards = len(self.topo.shards)
        # counted rendez-vous invariant: between rounds a worker's mailbox holds
        # n_shards (the completions of the previous round, not yet consumed)
        if self.mailbox is not None:
            self.mailbox.set(self.n_shards)
        if self.nvls:
            for key, ps in self.servers.items():
                goff, poff = self.worker.arena_offsets[ps.spec.task]
                ps.shard.round_bind_mc(self.arena.mcx, goff, poff, ps.spec.off, self.n_workers)
        elif fused:
            bufs = self._merge({self.worker_index: self.worker.buffer_handles()}
                               if self.worker else {})
            for key, ps in self.servers.items():
                for widx in range(self.n_workers):
                    g, p = bufs[widx][ps.spec.task]
                    ps.shard.round_bind(widx, g, p, ps.spec.off)
        self.worker_stream = torch.cuda.Stream(device=self.device)
        self.ps_stream = torch.cuda.Stream(device=self.device)
        # the shard whose kernel dominates a round (what a KernelTimer brackets)
        self.dominant = max(self.servers.values(), key=lambda ps: ps.spec.nelem,
                            default=None)
        self.seq = 0
        self._batches = {}
        self.staging = None
        self.h2d_stream = self.d2h_stream = self.pull_stream = None
        self.barrier()

    def _agree(self, err):
        """All ranks learn whether any of them failed; if so everyone tears its part
        down and raises NvlsUnavailable with the first failure's message."""
        import torch.distributed as dist
        errs = [err]
        if self.world > 1:
            errs = [None] * self.world
            dist.all_gather_object(errs, err)
        bad = [e for e in errs if e]
        if not bad:
            return
        if self.arena is not None:
            try:
                self.arena.destroy()
            except RuntimeError:
                pass
            self.arena = None
        for ps in self.servers.values():
            ps.close()
        self.servers.clear()
        raise NvlsUnavailable(bad[0])

    def _bcast(self, obj):
        import torch.distributed as dist
        box = [obj]
        if self.world > 1:
            dist.broadcast_object_list(box, src=0)
        return box[0]

    def _merge(self, mine):
        return merge_across_ranks(mine)

    def barrier(self):
        import torch
        import torch.distributed as dist
        torch.cuda.synchronize(self.device)
        if self.world > 1:
            dist.barrier()

    def set_variable(self, name, value):
        import numpy as np
        task, off, shape, numel = self.layout.entries[name]
        flat = np.ascontiguousarray(value, dtype=np.float32).reshape(-1)
        for key, ps in self.servers.items():
            spec = ps.spec
            if spec.task != task:
                continue
            lo, hi = max(off, spec.off), min(off + numel, spec.off + spec.nelem)
            if lo < hi:
                ps.shard.set_values(psx.VAR, flat[lo - off:hi - off], lo - spec.off)

    def _build_batch(self, mode):
        """The round as one psx_batch.  Counted rendez-vous: every wait compares
        with a constant (arrivals >= n_workers, mailbox >= n_shards) and the waiter
        consumes what it waited for, so the sequence is identical every round --
        replayable from a CUDA graph (capture_round)."""
        import ctypes
        ws, pss, wk = self.worker_stream, self.ps_stream, self.worker
        ops = []
        keep = []
        if wk is not None and self.fused:
            ids = (ctypes.c_uint64 * len(wk.clients))(*[c.id for c in wk.clients.values()])
            keep.append(ids)
            ops.append(dict(op=psx.OP_SIGNAL_COUNTED, ptr=ctypes.addressof(ids), n=len(ids),
                            id=self.mailbox.id, c=self.n_shards, stream=ws))
        elif wk is not None:
            ops.append(dict(op=psx.OP_MAILBOX_CONSUME, id=self.mailbox.id, c=self.n_shards,
                            stream=ws, uses_seq=False))
            for sp in wk.order:
                g = wk.grad_flat[sp.task]
                ops.append(dict(op=psx.OP_PUSH, id=wk.clients[sp.key].id,
                                ptr=g.data_ptr() + sp.off * g.element_size(), off=0,
                                n=sp.nelem, a=wk.wire, stream=ws))
        for ps in self.servers.values():
            ops.append(dict(op=psx.OP_ROUND_COUNTED if self.fused else psx.OP_APPLY_COUNTED,
                            id=ps.shard.id, a=mode, b=0, c=self.n_workers, stream=pss,
                            uses_seq=False))
        if wk is not None:
            ops.append(dict(op=psx.OP_MAILBOX_WAIT, id=self.mailbox.id, c=self.n_shards,
                            stream=ws, uses_seq=False))
        if wk is not None and not self.fused:
            for sp in wk.order:
                p = wk.param_flat[sp.task]
                ops.append(dict(op=psx.OP_PULL, id=wk.clients[sp.key].id,
                                ptr=p.data_ptr() + sp.off * p.element_size(), off=0,
                                n=sp.nelem, a=wk.wire, stream=ws, uses_seq=False))
        batch = psx.Batch(ops)
        batch.keep = keep
        return batch

    def _batch(self, mode):
        batch = self._batches.get(mode)
        if batch is None:
            batch = self._batches[mode] = self._build_batch(mode)
        return batch

    def round(self, mode, timer=None):
        """One global PS round, fully asynchronous: worker stream = signal/push ...
        wait/pull, PS stream = wait(arrival counter) + kernel; the GPUs' front
        ends do the ordering.  Synchronisation cost per rank and round is constant
        in the number of shards: one signal launch (fused) and one stream wait
        per hosted shard plus one on the worker's mailbox.  Without a timer the
        whole round is ONE call into libpsx (psx_batch)."""
        self.seq += 1
        if timer is None:
            self._batch(mode).run(self.seq)
            return
        ws, pss, wk = self.worker_stream, self.ps_stream, self.worker
        if wk is not None and self.fused:
            psx.signal_counted(list(wk.clients.values()), self.seq, self.mailbox,
                               self.n_shards, ws)
        elif wk is not None:
            self.mailbox.consume(self.n_shards, ws)
            wk.push(self.seq, ws)
        for ps in self.servers.values():
            timed = ps is self.dominant
            if timed:       # bracket the kernel alone: do the counted wait by hand first
                ps.shard.wait_arrivals(self.n_workers, pss)
                timer.start(pss)
            if self.fused:
                ps.shard.round_counted(mode, 0, self.n_workers, pss)
            else:
                ps.shard.apply_counted(mode, 0, self.n_workers, pss)
            if timed:
                timer.stop(pss)
        if wk is not None:
            self.mailbox.wait(self.n_shards, ws)
            if not self.fused:
                wk.pull(0, ws)

    def capture_round(self, mode, pre=None):
        """A CUDA graph holding ``pre()`` (e.g. the worker's forward/backward)
        followed by one PS round; ``graph.replay()`` then IS a training step.
        Launch-bound steps (the 318 KB MNIST model) are host-call bound otherwise."""
        import torch
        ws, pss = self.worker_stream, self.ps_stream
        batch = self._batch(mode)
        torch.cuda.synchronize(self.device)
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph, stream=ws):
            if pre is not None:
                pre()
            pss.wait_stream(ws)            # pull the PS stream into the capture
            # any non-zero sequence number: it only stamps the (unused here) slot
            # flags -- zero would mean "publish nothing"
            batch.run(1)
            ws.wait_stream(pss)            # and join it again
        return graph

    def round_host(self, mode):
        """The same round from HOST buffers, software-pipelined over the shards:
        while shard i's gradients cross PCIe (H2D stream), shard i-1 is pushed /
        applied / pulled and shard i-2's parameters go back to the host (D2H
        stream).  Five streams, so that no stage waits behind another stage's
        dependency: H2D, push, apply (PS), pull, D2H -- with pushes and pulls on
        ONE stream, pull(i) sat behind push(i+1), i.e. behind H2D(i+1), and the
        pipeline was one stage deeper than necessary (measured 18.5 ms = 18/16 of
        the PCIe duplex floor; (S+1)/S is the design point).
        Shards hosted by this rank skip the staging hop altogether: their gradients
        are DMA'd straight into this worker's landing slot and their parameters
        straight out of ``var`` (f32 wire).
        Every rank walks the shards in the SAME order: a shard's apply needs all W
        pushes, so it can only complete (and its pull / D2H start) when the slowest
        rank has reached it -- identical order makes that as early as possible, and
        the pushes are PCIe-paced (49 GB/s per rank), far below what incast into one
        NVLink port would need to matter.
        Returns once the round is enqueued: ``staging.grad`` and ``staging.param``
        belong to it until ``worker_stream`` has passed its end, so synchronise
        that stream before rewriting the gradients or reading the parameters."""
        import torch
        assert self.worker is not None and not self.fused, \
            "round_host runs on worker ranks of a staged-path cluster"
        if self.staging is None:
            self.staging = HostStaging(self.worker)
        if self.h2d_stream is None:
            self.h2d_stream = torch.cuda.Stream(device=self.device)
            self.d2h_stream = torch.cuda.Stream(device=self.device)
            self.pull_stream = torch.cuda.Stream(device=self.device)
            # direct DMA targets of the shards hosted here (f32 wire only: a bf16 slot
            # or parameter needs the casting kernels)
            self._direct = {}
            if self.worker.wire == psx.F32:
                for key, ps in self.servers.items():
                    n = ps.spec.nelem
                    self._direct[key] = (
                        psx.device_tensor(ps.shard.ptr(psx.SLOT0 + self.worker.index), n,
                                          torch.float32, self.device),
                        psx.device_tensor(ps.shard.ptr(psx.VAR), n, torch.float32, self.device))
        st, wk = self.staging, self.worker
        ws, pss, hs, ds, pl = (self.worker_stream, self.ps_stream, self.h2d_stream,
                               self.d2h_stream, self.pull_stream)
        self.seq += 1
        seq = self.seq
        hs.wait_stream(ws)                 # last round's pushes have read grad_flat
        hs.wait_stream(pss)                # ... and last round's applies their landing slots
        self.mailbox.consume(self.n_shards, ws)   # counted rendez-vous: start from zero
        pl.wait_stream(ds)                 # last round's D2H has read param_flat
        shards = self.topo.shards
        for sp in shards:
            host_g = st.grad[sp.task][sp.off:sp.off + sp.nelem]
            host_p = st.param[sp.task][sp.off:sp.off + sp.nelem]
            direct = self._direct.get(sp.key)
            # ---- gradients in
            with torch.cuda.stream(hs):
                if direct is not None:
                    direct[0].copy_(host_g, non_blocking=True)
                else:
                    g = wk.grad_flat[sp.task][sp.off:sp.off + sp.nelem]
                    g.copy_(host_g, non_blocking=True)
                ev = torch.cuda.Event()
                ev.record(hs)
            ws.wait_event(ev)
            if direct is not None:         # already in the slot: publish flag + arrival only
                wk.clients[sp.key].signal(seq, ws)
            else:
                wk.clients[sp.key].push(g.data_ptr(), sp.nelem, 0, wk.wire, seq, ws)
            # ---- apply (owner only)
            ps = self.servers.get(sp.key)
            if ps is not None:
                ps.shard.apply_counted(mode, 0, self.n_workers, pss)
            # ---- parameters out
            if direct is not None:
                wk.clients[sp.key].wait_applied(seq, pl)
                ev2 = torch.cuda.Event()
                ev2.record(pl)
                ds.wait_event(ev2)
                with torch.cuda.stream(ds):
                    host_p.copy_(direct[1], non_blocking=True)
            else:
                p = wk.param_flat[sp.task][sp.off:sp.off + sp.nelem]
                wk.clients[sp.key].pull(p.data_ptr(), sp.nelem, 0, wk.wire, seq, pl)
                ev2 = torch.cuda.Event()
                ev2.record(pl)
                ds.wait_event(ev2)
                with torch.cuda.stream(ds):
                    host_p.copy_(p, non_blocking=True)
        self.mailbox.wait(self.n_shards, ws)   # every shard applied (invariant restored)
        ws.wait_stream(ds)                 # the step ends when the host has the parameters
        ws.wait_stream(pl)

    def close(self):
        self.barrier()
        self._batches.clear()
        if self.worker is not None:
            self.worker.close()
        self.barrier()
        for ps in self.servers.values():
            ps.close()
        self.servers.clear()
        if self.mailbox is not None:
            self.mailbox.destroy()
        self.barrier()
        if self.arena is not None:
            self.arena.destroy()
            self.arena = None


class TensorListBinding(object):
    """A model's own (separate) tensors bound to their places in the PS buckets:
    ``push`` / ``pull`` move the whole list with ONE kernel launch per shard
    (psx_push_list / psx_pull_list, TMA-staged) instead of one copy per variable
    -- the reference issues one RecvTensor RPC per variable per direction."""

    def __init__(self, worker, tensors):
        """tensors: {variable name: contiguous float32 CUDA tensor of that shape}."""
        self.worker = worker
        self.keep = dict(tensors)              # keep the storages alive
        self.lists = OrderedDict()
        for spec in worker.topo.shards:
            ptrs, offs, counts = [], [], []
            for name, (task, off, shape, numel) in worker.layout.entries.items():
                if task != spec.task or name not in tensors:
                    continue
                t = tensors[name]
                assert t.is_contiguous() and t.numel() == numel and t.element_size() == 4, name
                lo, hi = max(off, spec.off), min(off + numel, spec.off + spec.nelem)
                if lo < hi:
                    ptrs.append(t.data_ptr() + (lo - off) * 4)
                    offs.append(lo - spec.off)
                    counts.append(hi - lo)
            if ptrs:
                self.lists[spec.key] = psx.TensorList(worker.clients[spec.key], ptrs, offs, counts)

    def push(self, seq=0, tma=True, stream=None):
        for lst in self.lists.values():
            lst.push(seq, tma, stream)

    def pull(self, wait_seq=0, tma=True, stream=None):
        for lst in self.lists.values():
            lst.pull(wait_seq, tma, stream)

    def close(self):
        for lst in self.lists.values():
            lst.destroy()
        self.lists.clear()
        self.keep.clear()
