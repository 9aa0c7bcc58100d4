"""The few TensorFlow entry points the reference's examples call, re-expressed
over the B200 engine, so that those scripts port line by line (SURVEY.md
appendix C).  Not a TensorFlow clone: tensors are torch tensors, the model's
forward/backward is ordinary torch code on the worker's GPU, and only the
PS-facing calls -- variable placement, push, optimizer apply, pull -- go through
libpsx.so.

    ClusterSpec / Server(...).join()     mnist_replica.py:85-95
    device(), constant(), Session.run    plus.py:23-33
    replica_device_setter, optimizers    engine.py
    ParameterClient                      the worker's session on the PS tasks:
        init_op / Supervisor chief-or-wait   mnist_replica.py:164-184
        sess.run([train_step, global_step])  mnist_replica.py:198-205
"""
import socket
import time
from contextlib import contextmanager

from . import endpoint, engine, psx
from .utils import bind_advertised
from .engine import (AdagradOptimizer, AdamOptimizer, GradientDescentOptimizer,  # noqa: F401
                     MomentumOptimizer, RMSPropOptimizer, replica_device_setter)


class ClusterSpec(object):
    """tf.train.ClusterSpec({'ps': [...], 'worker': [...]})."""

    def __init__(self, jobs):
        self.jobs = {k: list(v) for k, v in dict(jobs).items()}

    def get(self, name, default=None):
        return self.jobs.get(name, default)

    def job_tasks(self, name):
        return self.jobs[name]

    def __getitem__(self, name):
        return self.jobs[name]


class Server(object):
    """tf.train.Server(cluster, job_name=, task_index=): binds this task's
    address from the cluster spec; ``join()`` serves the endpoint for ever."""

    def __init__(self, cluster, job_name, task_index, gpus=0):
        if not isinstance(cluster, ClusterSpec):
            cluster = ClusterSpec(cluster)
        self.cluster, self.job_name, self.task_index = cluster, job_name, int(task_index)
        addr = cluster[job_name][self.task_index]
        self.target = 'grpc://%s' % addr
        port = int(addr.rsplit(':', 1)[1])
        self.listener = socket.socket()
        self.listener.setsockopt(socket.SOL_SOCKET, socket.SO_REUSEADDR, 1)
        bind_advertised(self.listener, port, addr.rsplit(':', 1)[0])
        self.endpoint = endpoint.Endpoint(job_name, self.task_index, cluster.jobs, gpus=gpus)

    def join(self):
        self.endpoint.serve(self.listener)


# ------------------------------------------------------------------ plus.py ----
_device_stack = [None]


@contextmanager
def device(name):
    """tf.device('/job:ps/task:0')."""
    job, task = name.strip('/').split('/')
    _device_stack.append((job.split(':')[1], int(task.split(':')[1])))
    try:
        yield
    finally:
        _device_stack.pop()


class Node(tuple):
    def __add__(self, other):
        return Node(('add', _device_stack[-1], self, other))


def constant(value):
    return Node(('const', _device_stack[-1], value))


class Session(object):
    """tf.Session(target): ``run(node)`` evaluates a (tiny) placed graph from the
    task behind ``target``; ``call`` runs a function inside that task."""

    def __init__(self, target):
        self.target = target

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        return False

    def run(self, node):
        return endpoint.call(self.target, 'eval', node=node)

    def call(self, fn, **kwargs):
        return endpoint.call(self.target, 'call', fn=fn, kwargs=kwargs)


# --------------------------------------------------------- worker-side session ---
class ParameterClient(object):
    """A worker task's session on the PS tasks of a cluster spec.

    variables: [(name, shape)] in creation order -> placed by
    replica_device_setter over len(cluster['ps']) tasks (or ``placement``).
    The chief (worker 0) runs the init_op; the others wait for it, like
    tf.train.Supervisor.prepare_or_wait_for_session (mnist_replica.py:166-184).
    """

    def __init__(self, cluster, variables, optimizer, worker_index, device=0,
                 placement=None, init=None, wire=psx.F32):
        import torch
        if not isinstance(cluster, ClusterSpec):
            cluster = ClusterSpec(cluster)
        self.cluster = cluster
        self.index = int(worker_index)
        self.n_workers = len(cluster['worker'])
        self.ps_addrs = cluster['ps']
        self.is_chief = self.index == 0
        self.device = device
        psx.init(device)
        self.layout = engine.VariableLayout(variables, len(self.ps_addrs), placement)
        ps_devices = [endpoint.call(a, 'device') for a in self.ps_addrs]
        # device ordinals on the PS side are irrelevant to the worker: it maps
        # the shard by handle; the topology only records one stripe per task
        self.topo = engine.Topology(self.layout, ps_devices,
                                    [device] * self.n_workers)
        hyper = optimizer.hyper
        handles = {}
        for spec in self.topo.shards:
            handles[spec.key] = endpoint.call(
                self.ps_addrs[spec.task], 'create_shard', key=spec.key, nelem=spec.nelem,
                opt=optimizer.opt, hyper=hyper, n_slots=self.n_workers, wire=wire)
        self.worker = engine.Worker(self.index, self.topo, handles, wire=wire)
        for key, h in self.worker.client_handles().items():
            endpoint.call(self.ps_addrs[key[0]], 'register_client', key=key,
                          slot=self.index, handle=h)
        self.params, self.grads = self.worker.params, self.worker.grads
        self.stream = torch.cuda.Stream(device=device)
        self.push_seq = 0
        self.serving = None           # (mode, replicas_to_aggregate) once the PS loops run
        # global_step as mirrored into this worker's HBM by the apply that consumed
        # its push, copied to pinned host memory on the stream (never a request)
        self._step_host = torch.zeros(1, dtype=torch.int64).pin_memory()
        self._step_event = None
        self._step_client = self.worker.clients[self.topo.shards[0].key]
        # PS endpoints running as threads of THIS process (tests, notebooks): stream
        # waits on a shard served in-process can deadlock (psx.h, psx_client_poll), so
        # such a session waits on the host instead
        self.in_process = any(c.poll()["in_process"] for c in self.worker.clients.values())
        if self.is_chief:
            for name, value in (init or {}).items():
                self.assign(name, value)
            for a in self.ps_addrs:
                endpoint.call(a, 'put', name='initialized', value=True)
        else:
            for a in self.ps_addrs:
                deadline = time.time() + 300
                while not endpoint.call(a, 'get', name='initialized', default=False):
                    if time.time() > deadline:
                        raise RuntimeError('chief never initialised the variables')
                    time.sleep(0.05)
        self._last_step = self.global_step()
        self.pull()

    def assign(self, name, value):
        import numpy as np
        task, off, shape, numel = self.layout.entries[name]
        flat = np.ascontiguousarray(value, dtype=np.float32).reshape(-1)
        assert flat.size == numel
        endpoint.call(self.ps_addrs[task], 'set_values', key=(task, 0), which=psx.VAR,
                      off=off, data=flat.tobytes())

    def read(self, name):
        import numpy as np
        task, off, shape, numel = self.layout.entries[name]
        raw = endpoint.call(self.ps_addrs[task], 'get_values', key=(task, 0), which=psx.VAR,
                            off=off, n=numel)
        return np.frombuffer(raw, np.float32).reshape(shape).copy()

    def _enqueue_pull(self):
        for spec in self.topo.shards:
            p = self.worker.param_flat[spec.task]
            self.worker.clients[spec.key].pull(p.data_ptr() + spec.off * p.element_size(),
                                               spec.nelem, 0, self.worker.wire, 0, self.stream)

    def pull(self):
        """PULL (Variable reads of the next sess.run), synchronously."""
        self._enqueue_pull()
        self.stream.synchronize()

    def _serve(self, mode, aggregate):
        """First step only: make sure every PS shard runs its serving loop in this
        discipline (one request per PS task, then never again)."""
        want = (int(mode), int(aggregate))
        if self.serving is None:
            for spec in self.topo.shards:
                endpoint.call(self.ps_addrs[spec.task], 'serve', key=spec.key, mode=want[0],
                              replicas_to_aggregate=want[1])
            self.serving = want
        elif self.serving != want:
            raise RuntimeError('this session already trains with mode/aggregate %r' %
                               (self.serving,))

    def _known_step(self):
        """The newest global_step the host has seen (waits for the last enqueued
        8-byte copy only if it has not landed yet -- normally it has)."""
        if self._step_event is not None:
            self._step_event.synchronize()
            self._step_event = None
            self._last_step = int(self._step_host[0])
        return self._last_step

    def minimize(self, mode=psx.MODE_ASYNC_ORDERED, replicas_to_aggregate=None, fetch_step=True):
        """One ``sess.run([train_step, global_step])`` (mnist_replica.py:204) with NO
        request to the PS: PUSH this worker's gradients into its landing slots (the
        kernel's epilogue bumps each shard's arrival counter), stream-wait until the
        PS's serving loop has consumed the push, PULL.  The PS applies pushes as
        they arrive (async, the reference's default), or -- ``mode=MODE_SYNC_MEAN``
        -- runs SyncReplicasOptimizer on the device: the first
        ``replicas_to_aggregate`` fresh gradients by ARRIVAL are averaged and
        applied, later / stale ones dropped, every worker released by a token
        (mnist_replica.py:109-113,148-162).

        Returns global_step.  fetch_step=True waits for the 8-byte copy of the step
        this push produced (the value TF returns); fetch_step=False never blocks the
        host and returns the newest step already known (one step behind)."""
        import torch
        if mode == psx.MODE_SUM:
            raise ValueError('the serving loop applies per push (async) or averages (sync)')
        aggregate = self.n_workers if replicas_to_aggregate is None \
            else max(1, min(int(replicas_to_aggregate), self.n_workers))
        self._serve(mode, aggregate if mode == psx.MODE_SYNC_MEAN else 1)
        stamp = self._known_step()              # the step our parameters are at
        cur = torch.cuda.current_stream(self.device)
        self.stream.wait_stream(cur)
        self.push_seq += 1
        wk = self.worker
        for spec in wk.order:
            g = wk.grad_flat[spec.task]
            wk.clients[spec.key].push_stamped(g.data_ptr() + spec.off * g.element_size(),
                                              spec.nelem, 0, wk.wire, self.push_seq, stamp,
                                              self.stream)
        what = "tokens" if mode == psx.MODE_SYNC_MEAN else "applied"
        for spec in self.topo.shards:
            if self.in_process:
                self.stream.synchronize()          # the push has left ...
                wk.clients[spec.key].wait_host(what, self.push_seq)   # ... and was consumed
            elif mode == psx.MODE_SYNC_MEAN:
                wk.clients[spec.key].wait_tokens(self.push_seq, self.stream)
            else:
                wk.clients[spec.key].wait_applied(self.push_seq, self.stream)
        self._enqueue_pull()
        self._step_client.read_step_async(self._step_host.data_ptr(), self.stream)
        self._step_event = torch.cuda.Event()
        self._step_event.record(self.stream)
        cur.wait_stream(self.stream)            # the next forward reads the pulled parameters
        if fetch_step:
            return self._known_step()
        return self._last_step

    def global_step(self):
        st = endpoint.call(self.ps_addrs[0], 'state', key=(0, 0))
        return st['global_step']

    def save(self, path):
        """Checkpoint every PS task's shards (what the chief's Supervisor does
        with its logdir, mnist_replica.py:165-170); returns the files written."""
        return [endpoint.call(a, 'save', path=path) for a in self.ps_addrs]

    def restore(self, path):
        files = [endpoint.call(a, 'restore', path=path) for a in self.ps_addrs]
        self._step_event = None
        self._last_step = self.global_step()
        self.pull()
        return files

    def close(self):
        """Detach from every PS task first (they stop publishing into this worker's
        client blocks and drain), only then free the blocks."""
        import torch
        self.stream.synchronize()
        torch.cuda.synchronize(self.device)
        for spec in self.topo.shards:
            try:
                endpoint.call(self.ps_addrs[spec.task], 'unregister_client', key=spec.key,
                              slot=self.index)
            except (OSError, RuntimeError, EOFError, AssertionError):
                pass                      # the PS task is already gone (cluster tear-down)
        self.worker.close()
