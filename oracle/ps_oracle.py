"""numpy restatement of the reference's PS data path.  TEST INFRASTRUCTURE ONLY.

Only ``tests/``, ``__graft_entry__.smoke()`` and ``bench.py``'s CPU legs may
import this module; nothing under ``tfmesos_b200/`` does.

PARITY UNPINNED upstream: douban/tfmesos has no tests and no golden vectors for
this path (``tox.ini:8``); the arithmetic belongs to TensorFlow 0.12
(``requirements.txt:10``), absent from ``/root/reference`` and not installable
here.  This file restates TF 0.12's published ``ApplyGradientDescent`` /
``ApplyAdam`` / ``replica_device_setter`` behaviour, anchored on the reference's
call sites (cited per function), and is itself pinned by hand-computed
known-answer tests (``tests/test_oracle_kat.py``) and by agreement with the
independent C restatement ``oracle/ps_oracle.c``.

Every array op below is float32 with one rounding per operation (numpy never
fuses a*b+c), i.e. the same value sequence as the C file and the CUDA kernels.
"""
from __future__ import annotations

import ctypes
import os
import subprocess
import tempfile

import numpy as np

F = np.float32

ASYNC_ORDERED, SUM, SYNC_MEAN = 0, 1, 2
SGD, ADAM = 0, 1

HERE = os.path.dirname(os.path.abspath(__file__))


# --------------------------------------------------------------------------
# placement: tf.train.replica_device_setter   (mnist.py:43, mnist_replica.py:116)
# --------------------------------------------------------------------------
def replica_device_setter_placement(variable_names, ps_tasks):
    """Round-robin, per Variable op, in creation order, starting at task 0.

    Slot variables (Adam m/v, beta powers) are created under colocate_with and
    never advance the counter (SURVEY.md appendix A.1).  Returns
    ``{name: ps_task_index}`` in creation order.
    """
    if ps_tasks <= 0:
        return {name: None for name in variable_names}
    return {name: i % ps_tasks for i, name in enumerate(variable_names)}


MNIST_SOFTMAX_VARS = ["W", "b", "global_step"]                      # mnist.py:44-46
MNIST_MLP_VARS = ["global_step", "hid_w", "hid_b", "sm_w", "sm_b"]  # mnist_replica.py:121-134
NMF_PLACEMENT = {"W": 0, "H": 1}                                    # matrix_factorization.py:21-28


# --------------------------------------------------------------------------
# optimizer applies
# --------------------------------------------------------------------------
def sgd_apply(var, g, lr):
    """ApplyGradientDescent (mnist.py:55, matrix_factorization.py:39-41)."""
    var -= g * F(lr)
    return var


def adam_alpha(lr, b1p, b2p):
    return (F(lr) * np.sqrt(F(1) - F(b2p), dtype=F)) / (F(1) - F(b1p))


def adam_apply(var, m, v, g, lr, b1, b2, eps, b1p, b2p):
    """ApplyAdam with the stored powers (mnist_replica.py:147); eps outside."""
    alpha = adam_alpha(lr, b1p, b2p)
    m += (g - m) * (F(1) - F(b1))
    v += (g * g - v) * (F(1) - F(b2))
    var -= (m * alpha) / (np.sqrt(v, dtype=F) + F(eps))
    return var, m, v


class Shard:
    """One PS task's state for a flat bucket of variables."""

    def __init__(self, nelem, opt=SGD, lr=0.01, b1=0.9, b2=0.999, eps=1e-8):
        self.n = int(nelem)
        self.opt = opt
        self.lr, self.b1, self.b2, self.eps = F(lr), F(b1), F(b2), F(eps)
        self.var = np.zeros(self.n, F)
        self.m = np.zeros(self.n, F)
        self.v = np.zeros(self.n, F)
        self.b1p, self.b2p = F(b1), F(b2)     # initialised to beta, A.3
        self.step = 0                          # global_step

    def _apply(self, g):
        if self.opt == SGD:
            sgd_apply(self.var, g, self.lr)
        else:
            adam_apply(self.var, self.m, self.v, g, self.lr, self.b1, self.b2,
                       self.eps, self.b1p, self.b2p)
            self.b1p = F(self.b1p * self.b1)
            self.b2p = F(self.b2p * self.b2)
        self.step += 1

    def round(self, slots, mode):
        """slots: [W, n] float32, applied under discipline ``mode``."""
        slots = np.asarray(slots, F)
        W = slots.shape[0]
        if mode == ASYNC_ORDERED:
            for w in range(W):
                self._apply(slots[w])
            return
        acc = slots[0].copy()
        for w in range(1, W):
            acc = acc + slots[w]
        if mode == SYNC_MEAN:
            acc = acc / F(W)
        self._apply(acc)


def rows_round(shard, row_len, idx_lists, row_lists, mode):
    """Index-list (IndexedSlices) round on a :class:`Shard` viewed as
    [n / row_len, row_len] (SURVEY 8f-3; reference: the NMF row blocks of
    examples/matrix_factorization.py:21-28,43-49).  idx_lists[w]: strictly
    ascending row indices of worker w; row_lists[w]: [k_w, row_len] gradients.
    A row pushed by several workers gets ((g_w + g_w') + ...) in worker order;
    SYNC_MEAN divides by the number of workers; SGD / Adam are applied ONCE to
    every touched row, untouched rows keep var / m / v; beta powers and
    global_step advance once."""
    assert mode in (SUM, SYNC_MEAN)
    W = len(idx_lists)
    var = shard.var.reshape(-1, row_len)
    m = shard.m.reshape(-1, row_len)
    v = shard.v.reshape(-1, row_len)
    acc = {}
    for w in range(W):
        idx = np.asarray(idx_lists[w], np.int64)
        assert np.all(np.diff(idx) > 0), "indices must be strictly ascending"
        for k, r in enumerate(idx):
            g = np.asarray(row_lists[w][k], F)
            acc[int(r)] = g.copy() if int(r) not in acc else (acc[int(r)] + g).astype(F)
    alpha = adam_alpha(shard.lr, shard.b1p, shard.b2p) if shard.opt == ADAM else None
    for r, g in acc.items():
        if mode == SYNC_MEAN:
            g = (g / F(W)).astype(F)
        if shard.opt == SGD:
            var[r] -= g * shard.lr
        else:
            m[r] += (g - m[r]) * (F(1) - shard.b1)
            v[r] += (g * g - v[r]) * (F(1) - shard.b2)
            var[r] -= (m[r] * alpha) / (np.sqrt(v[r], dtype=F) + shard.eps)
    if shard.opt == ADAM:
        shard.b1p = F(shard.b1p * shard.b1)
        shard.b2p = F(shard.b2p * shard.b2)
    shard.step += 1


# --------------------------------------------------------------------------
# bf16 wire format
# --------------------------------------------------------------------------
def f32_to_bf16(x):
    u = np.asarray(x, F).view(np.uint32).astype(np.uint64)
    nan = (u & 0x7FFFFFFF) > 0x7F800000
    lsb = (u >> 16) & 1
    r = ((u + 0x7FFF + lsb) >> 16).astype(np.uint16)
    r[nan] = ((u[nan] >> 16) | 0x40).astype(np.uint16)
    return r


def bf16_to_f32(h):
    return (np.asarray(h, np.uint16).astype(np.uint32) << 16).view(F)


# --------------------------------------------------------------------------
# model maths (closed-form gradients, SURVEY.md A.6); float32 throughout
# --------------------------------------------------------------------------
def _softmax(z):
    z = z - z.max(axis=1, keepdims=True)
    e = np.exp(z, dtype=F)
    return e / e.sum(axis=1, keepdims=True)


def softmax_regression_grads(W, b, x, y_):
    """mnist.py:48-50: L = -sum(y_*log(softmax(xW+b))), no clipping."""
    p = _softmax(x @ W + b)
    loss = -np.sum(y_ * np.log(p, dtype=F), dtype=F)
    d = p - y_
    return loss, x.T @ d, d.sum(axis=0)


def mlp_grads(hid_w, hid_b, sm_w, sm_b, x, y_):
    """mnist_replica.py:140-145: relu MLP, L = -sum(y_*log(clip(p,1e-10,1)))."""
    lin = x @ hid_w + hid_b
    h = np.maximum(lin, F(0))
    p = _softmax(h @ sm_w + sm_b)
    pc = np.clip(p, F(1e-10), F(1.0))
    loss = -np.sum(y_ * np.log(pc, dtype=F), dtype=F)
    inside = ((p >= F(1e-10)) & (p <= F(1.0))).astype(F)
    dp = -(y_ / pc) * inside                       # dL/dp through clip
    dz = p * (dp - np.sum(dp * p, axis=1, keepdims=True))
    d_sm_w = h.T @ dz
    d_sm_b = dz.sum(axis=0)
    dh = dz @ sm_w.T
    dlin = dh * (lin > 0).astype(F)
    return loss, x.T @ dlin, dlin.sum(axis=0), d_sm_w, d_sm_b


NMF_INFINITY = F(10e12)                            # matrix_factorization.py:10


def nmf_grads(W, H, R):
    """matrix_factorization.py:30-36: L = |R-WH|_F^2 + 1e13*(sum(|W|-W)+sum(|H|-H))."""
    E = R - W @ H
    loss = np.sum(E * E, dtype=F) + NMF_INFINITY * (
        np.sum(np.abs(W) - W, dtype=F) + np.sum(np.abs(H) - H, dtype=F))
    dW = F(-2) * (E @ H.T) + NMF_INFINITY * (np.sign(W) - F(1))
    dH = F(-2) * (W.T @ E) + NMF_INFINITY * (np.sign(H) - F(1))
    return loss, dW.astype(F), dH.astype(F)


def truncated_normal(rng, shape, stddev):
    """tf.truncated_normal: resample beyond 2 sigma (mnist_replica.py:124-133)."""
    out = rng.standard_normal(shape)
    bad = np.abs(out) > 2.0
    while bad.any():
        out[bad] = rng.standard_normal(int(bad.sum()))
        bad = np.abs(out) > 2.0
    return (out * stddev).astype(F)


# --------------------------------------------------------------------------
# C restatement loader (oracle/ps_oracle.c -> oracle/_build/libps_oracle.so)
# --------------------------------------------------------------------------
_LIB = None


def build_c(force=False):
    out_dir = os.path.join(HERE, "_build")
    so = os.path.join(out_dir, "libps_oracle.so")
    src = os.path.join(HERE, "ps_oracle.c")
    if force or not os.path.exists(so) or os.path.getmtime(so) < os.path.getmtime(src):
        try:
            os.makedirs(out_dir, exist_ok=True)
        except OSError:
            pass
        if not os.access(out_dir, os.W_OK):
            # a read-only tree (e.g. a benchmark run from an installed checkout):
            # build beside it, never into it
            so = os.path.join(tempfile.mkdtemp(prefix="ps_oracle_"), "libps_oracle.so")
        subprocess.check_call(
            ["gcc", "-O2", "-std=c11", "-ffp-contract=off", "-fno-fast-math",
             "-fPIC", "-shared", src, "-o", so, "-lm", "-lpthread"])
    return so


def c_lib():
    global _LIB
    if _LIB is not None:
        return _LIB
    lib = ctypes.CDLL(build_c())
    fp = ctypes.POINTER(ctypes.c_float)
    sz = ctypes.c_size_t
    fl = ctypes.c_float
    lib.psx_oracle_sgd.argtypes = [fp, fp, sz, fl]
    lib.psx_oracle_sgd.restype = None
    lib.psx_oracle_adam_alpha.argtypes = [fl, fl, fl]
    lib.psx_oracle_adam_alpha.restype = fl
    lib.psx_oracle_adam.argtypes = [fp, fp, fp, fp, sz, fl, fl, fl, fl, fl, fl]
    lib.psx_oracle_adam.restype = None
    i64p = ctypes.POINTER(ctypes.c_int64)
    lib.psx_oracle_round_sgd.argtypes = [fp, fp, sz, ctypes.c_int, sz, fl,
                                         ctypes.c_int, fp, i64p]
    lib.psx_oracle_round_sgd.restype = ctypes.c_int
    lib.psx_oracle_round_adam.argtypes = [fp, fp, fp, fp, sz, ctypes.c_int, sz,
                                          fl, fl, fl, fl, ctypes.c_int, fp, fp, i64p]
    lib.psx_oracle_round_adam.restype = ctypes.c_int
    lib.psx_oracle_f32_to_bf16.argtypes = [fl]
    lib.psx_oracle_f32_to_bf16.restype = ctypes.c_uint16
    lib.psx_oracle_bf16_to_f32.argtypes = [ctypes.c_uint16]
    lib.psx_oracle_bf16_to_f32.restype = fl
    u16p = ctypes.POINTER(ctypes.c_uint16)
    lib.psx_oracle_cast_f32_bf16.argtypes = [u16p, fp, sz]
    lib.psx_oracle_cast_f32_bf16.restype = None
    lib.psx_oracle_cast_bf16_f32.argtypes = [fp, u16p, sz]
    lib.psx_oracle_cast_bf16_f32.restype = None
    i64pp = ctypes.POINTER(ctypes.POINTER(ctypes.c_int64))
    lib.psx_oracle_rows_round.argtypes = [fp, fp, fp, sz, sz, ctypes.c_int, i64pp,
                                          ctypes.POINTER(fp), ctypes.POINTER(sz), ctypes.c_int,
                                          ctypes.c_int, fl, fl, fl, fl, fl, fl, fp]
    lib.psx_oracle_rows_round.restype = ctypes.c_int
    lib.psx_oracle_threads.restype = ctypes.c_int
    fpp = ctypes.POINTER(fp)
    lib.psx_oracle_cpu_ps_round.argtypes = [fp, fp, fp, fp, sz, fpp, fpp,
                                            ctypes.c_int, sz, ctypes.c_int, fl, fl,
                                            fl, fl, ctypes.c_int, fp, fp, i64p,
                                            ctypes.c_int]
    lib.psx_oracle_cpu_ps_round.restype = ctypes.c_int
    lib.psx_oracle_cpu_ps_init.argtypes = [fp, fp, fp, fp, sz, fpp, fpp, ctypes.c_int, sz, fp]
    lib.psx_oracle_cpu_ps_init.restype = ctypes.c_int
    lib.psx_oracle_pool_start.argtypes = [ctypes.c_int]
    lib.psx_oracle_pool_start.restype = ctypes.c_int
    lib.psx_oracle_pool_threads.restype = ctypes.c_int
    lib.psx_oracle_pool_stop.restype = None
    _LIB = lib
    return lib


def _fp(a):
    assert a.dtype == F and a.flags.c_contiguous
    return a.ctypes.data_as(ctypes.POINTER(ctypes.c_float))


class CShard:
    """Same interface as :class:`Shard`, arithmetic done by ps_oracle.c."""

    def __init__(self, nelem, opt=SGD, lr=0.01, b1=0.9, b2=0.999, eps=1e-8):
        self.lib = c_lib()
        self.n = int(nelem)
        self.opt = opt
        self.hyper = (float(F(lr)), float(F(b1)), float(F(b2)), float(F(eps)))
        self.var = np.zeros(self.n, F)
        self.m = np.zeros(self.n, F)
        self.v = np.zeros(self.n, F)
        self.state = np.array([b1, b2], F)
        self._step = ctypes.c_int64(0)
        self.scratch = np.zeros(self.n, F)

    @property
    def step(self):
        return self._step.value

    @property
    def b1p(self):
        return self.state[0]

    @property
    def b2p(self):
        return self.state[1]

    def round(self, slots, mode):
        slots = np.ascontiguousarray(slots, F)
        W, n = slots.shape
        assert n == self.n
        lr, b1, b2, eps = self.hyper
        if self.opt == SGD:
            rc = self.lib.psx_oracle_round_sgd(
                _fp(self.var), _fp(slots), n, W, n, lr, mode, _fp(self.scratch),
                ctypes.byref(self._step))
        else:
            rc = self.lib.psx_oracle_round_adam(
                _fp(self.var), _fp(self.m), _fp(self.v), _fp(slots), n, W, n, lr,
                b1, b2, eps, mode, _fp(self.state), _fp(self.scratch),
                ctypes.byref(self._step))
        assert rc == 0, rc


def cpu_quota_cores(root="/sys/fs/cgroup"):
    """CPU bandwidth the container may use, in cores (cgroup v2 ``cpu.max`` or v1
    ``cpu.cfs_quota_us / cpu.cfs_period_us``); None when unlimited.  The pool's GPU
    boxes show 128 CPUs but run their containers under a 16-core CFS quota: 128
    busy threads exhaust it within each 100 ms period and are throttled until the
    next one -- the "bimodal" 7 ms / 100 ms rounds of profiles/r22-r29
    (``nr_throttled`` climbs, profiles/r30).  A pool of exactly `quota` threads is
    never throttled: 15.0 +- 0.1 ms for the same round."""
    try:
        txt = open(os.path.join(root, "cpu.max")).read().split()
        if txt and txt[0] != "max":
            return float(txt[0]) / float(txt[1])
        if txt:
            return None
    except (OSError, ValueError, IndexError):
        pass
    try:
        q = int(open(os.path.join(root, "cpu", "cpu.cfs_quota_us")).read())
        p = int(open(os.path.join(root, "cpu", "cpu.cfs_period_us")).read())
        if q > 0 and p > 0:
            return q / float(p)
    except (OSError, ValueError):
        pass
    return None


def usable_threads():
    """Threads worth running: the CPUs this process may be scheduled on, capped by
    the container's CPU quota."""
    n = len(os.sched_getaffinity(0))
    q = cpu_quota_cores()
    if q is not None:
        n = max(1, min(n, int(q)))
    return n


def c_rows_round(shard, row_len, idx_lists, row_lists, mode):
    """:func:`rows_round` by ps_oracle.c (the second restatement) on a :class:`CShard`."""
    assert mode in (SUM, SYNC_MEAN)
    lib = c_lib()
    W = len(idx_lists)
    idx = [np.ascontiguousarray(i, np.int64) for i in idx_lists]
    rows = [np.ascontiguousarray(r, F).reshape(-1, row_len) for r in row_lists]
    i64p = ctypes.POINTER(ctypes.c_int64)
    fp = ctypes.POINTER(ctypes.c_float)
    pi = (i64p * W)(*[a.ctypes.data_as(i64p) for a in idx])
    pr = (fp * W)(*[a.ctypes.data_as(fp) for a in rows])
    k = (ctypes.c_size_t * W)(*[a.size for a in idx])
    lr, b1, b2, eps = shard.hyper
    scratch = np.zeros(row_len, F)
    rc = lib.psx_oracle_rows_round(_fp(shard.var), _fp(shard.m), _fp(shard.v),
                                   shard.n // row_len, row_len, W, pi, pr, k,
                                   int(shard.opt == ADAM), int(mode == SYNC_MEAN), lr, b1, b2, eps,
                                   float(shard.state[0]), float(shard.state[1]), _fp(scratch))
    assert rc == 0, "indices must be strictly ascending and inside the matrix"
    if shard.opt == ADAM:
        shard.state[0] = F(shard.state[0] * F(b1))
        shard.state[1] = F(shard.state[1] * F(b2))
    shard._step.value += 1


class CpuPsBaseline:
    """Multi-threaded CPU-PS round (memcpy push, apply, memcpy pull) used as the
    timed CPU baseline by bench.py.  The arrays come untouched from the
    allocator and are FIRST-TOUCHED by the pool thread that owns each range in
    every later round (psx_oracle_cpu_ps_init), so NUMA placement is the same on
    every run; the pool is persistent, its threads are pinned, and it is sized to
    the container's CPU quota (usable_threads)."""

    def __init__(self, nelem, W, opt=ADAM, lr=0.01, b1=0.9, b2=0.999, eps=1e-8,
                 threads=0):
        self.lib = c_lib()
        self.n, self.W, self.opt = int(nelem), int(W), opt
        self.hyper = (float(F(lr)), float(F(b1)), float(F(b2)), float(F(eps)))
        # threads = 0: as many as the container can actually run (affinity capped by
        # its CPU quota)
        self.threads = self.lib.psx_oracle_pool_start(int(threads) if threads else usable_threads())
        assert self.threads > 0, "thread pool failed to start (%d)" % self.threads
        self.var = np.empty(self.n, F)           # np.empty: pages not touched yet
        self.m = np.empty(self.n, F)
        self.v = np.empty(self.n, F)
        self.slots = np.empty((self.W, self.n), F)
        self.scratch = np.empty(self.n, F)
        self.grads = [np.empty(self.n, F) for _ in range(self.W)]
        self.params = [np.empty(self.n, F) for _ in range(self.W)]
        self.state = np.array([b1, b2], F)
        self._step = ctypes.c_int64(0)
        fp = ctypes.POINTER(ctypes.c_float)
        self._g = (fp * self.W)(*[_fp(g) for g in self.grads])
        self._p = (fp * self.W)(*[_fp(p) for p in self.params])
        rc = self.lib.psx_oracle_cpu_ps_init(
            _fp(self.var), _fp(self.m), _fp(self.v), _fp(self.slots), self.n, self._g,
            self._p, self.W, self.n, _fp(self.scratch))
        assert rc > 0, rc

    def round(self, mode=SUM, threads=0):
        lr, b1, b2, eps = self.hyper
        rc = self.lib.psx_oracle_cpu_ps_round(
            _fp(self.var), _fp(self.m), _fp(self.v), _fp(self.slots), self.n,
            self._g, self._p, self.W, self.n, int(self.opt == ADAM), lr, b1, b2,
            eps, mode, _fp(self.state), _fp(self.scratch),
            ctypes.byref(self._step), threads)
        assert rc > 0, rc
        return rc
