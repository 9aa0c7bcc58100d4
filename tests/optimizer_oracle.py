"""Two CPU restatements of the Momentum / Adagrad / RMSProp updates of the PS data
plane (TF r0.12 ``ApplyMomentum`` / ``ApplyAdagrad`` / ``ApplyRMSProp``, and their
``SparseApply*`` counterparts for index-list rows).  Test infrastructure only.

The numpy :class:`Shard` and the C :class:`CShard` (``optimizer_oracle.c``) share
the interface of ``oracle.ps_oracle.Shard`` / ``CShard`` -- ``var``, ``m``, ``v``,
``step``, ``round(slots, mode)`` -- so the GPU tests compare the kernels against
them the way the SGD / Adam tests compare against the shared oracle, which stays
the reference for those two.  Every array op is float32 with one rounding per
operation (numpy never fuses a*b+c; the C file is compiled with
-ffp-contract=off).

hyper is the shard header's {lr, b1, b2, eps}; per optimizer it means
``{lr, momentum}``, ``{lr, initial_accumulator_value}`` and
``{lr, decay, momentum, epsilon}``.  Initial state: Momentum accum = 0, Adagrad
accum = initial_accumulator_value, RMSProp ms = 1 and mom = 0.
"""
import ctypes
import os
import subprocess
import tempfile

import numpy as np

F = np.float32
ASYNC_ORDERED, SUM, SYNC_MEAN = 0, 1, 2
MOMENTUM, ADAGRAD, RMSPROP = 2, 3, 4
OPTS = (MOMENTUM, ADAGRAD, RMSPROP)
NAMES = {MOMENTUM: "momentum", ADAGRAD: "adagrad", RMSPROP: "rmsprop"}
STATE_ARRAYS = {MOMENTUM: 1, ADAGRAD: 1, RMSPROP: 2}
# hyper-parameters the tests use by default: TF's defaults where TF has them
DEFAULT_HYPER = {MOMENTUM: (0.01, 0.9, 0.0, 0.0), ADAGRAD: (0.01, 0.1, 0.0, 0.0),
                 RMSPROP: (0.01, 0.9, 0.5, 1e-10)}

HERE = os.path.dirname(os.path.abspath(__file__))


def initial_state(opt, hyper, n):
    """(m, v) as a freshly created shard holds them."""
    m0 = {MOMENTUM: 0.0, ADAGRAD: hyper[1], RMSPROP: 1.0}[opt]
    return np.full(n, F(m0), F), np.zeros(n, F)


def apply(opt, var, m, v, g, hyper):
    """One update of ``var`` (and the state arrays) in place by gradient ``g``."""
    lr, b1, b2, eps = (F(h) for h in hyper)
    if opt == MOMENTUM:
        m *= b1
        m += g
        var -= m * lr
    elif opt == ADAGRAD:
        m += g * g
        var -= (g * lr) * (F(1) / np.sqrt(m, dtype=F))
    elif opt == RMSPROP:
        m += (g * g - m) * (F(1) - b1)
        v *= b2
        v += (g * lr) / np.sqrt(m + eps, dtype=F)
        var -= v
    else:
        raise ValueError("unknown optimizer %r" % (opt,))


class Shard(object):
    """numpy restatement: one PS shard of ``nelem`` elements."""

    def __init__(self, nelem, opt, hyper=None):
        self.n, self.opt = int(nelem), opt
        self.hyper = tuple(float(F(h)) for h in (hyper or DEFAULT_HYPER[opt]))
        self.var = np.zeros(self.n, F)
        self.m, self.v = initial_state(opt, self.hyper, self.n)
        self.step = 0

    def round(self, slots, mode):
        slots = np.asarray(slots, F)
        if mode == ASYNC_ORDERED:
            for g in slots:
                apply(self.opt, self.var, self.m, self.v, g, self.hyper)
                self.step += 1
            return
        acc = slots[0].copy()
        for g in slots[1:]:
            acc = acc + g
        if mode == SYNC_MEAN:
            acc = acc / F(slots.shape[0])
        apply(self.opt, self.var, self.m, self.v, acc, self.hyper)
        self.step += 1


def rows_round(shard, row_len, idx_lists, row_lists, mode):
    """Index-list round on a :class:`Shard` viewed as [n / row_len, row_len]: the
    rows of every worker summed in worker order, / W for SYNC_MEAN, one update per
    touched row; untouched rows keep var and state; global_step advances once."""
    assert mode in (SUM, SYNC_MEAN)
    W = len(idx_lists)
    var, m, v = (a.reshape(-1, row_len) for a in (shard.var, shard.m, shard.v))
    acc = {}
    for w in range(W):
        idx = np.asarray(idx_lists[w], np.int64)
        assert np.all(np.diff(idx) > 0), "indices must be strictly ascending"
        for k, r in enumerate(idx):
            g = np.asarray(row_lists[w][k], F)
            acc[int(r)] = g.copy() if int(r) not in acc else (acc[int(r)] + g).astype(F)
    for r, g in acc.items():
        if mode == SYNC_MEAN:
            g = (g / F(W)).astype(F)
        apply(shard.opt, var[r], m[r], v[r], g, shard.hyper)
    shard.step += 1


# ------------------------------------------------------------------ C side ----
_LIB = None


def c_lib():
    """optimizer_oracle.c, compiled once per process into a temporary directory
    (the tree may be read-only)."""
    global _LIB
    if _LIB is None:
        so = os.path.join(tempfile.mkdtemp(prefix="optimizer_oracle_"), "liboptimizer_oracle.so")
        subprocess.check_call(
            ["gcc", "-O2", "-std=c11", "-ffp-contract=off", "-fno-fast-math", "-fPIC",
             "-shared", os.path.join(HERE, "optimizer_oracle.c"), "-o", so, "-lm"])
        lib = ctypes.CDLL(so)
        fp = ctypes.POINTER(ctypes.c_float)
        sz, i32 = ctypes.c_size_t, ctypes.c_int
        i64p = ctypes.POINTER(ctypes.c_int64)
        lib.opt_oracle_round.argtypes = [i32, fp, fp, fp, fp, sz, i32, sz, fp, i32, fp, i64p]
        lib.opt_oracle_round.restype = i32
        lib.opt_oracle_rows_round.argtypes = [i32, fp, fp, fp, sz, sz, i32,
                                              ctypes.POINTER(i64p), ctypes.POINTER(fp),
                                              ctypes.POINTER(sz), i32, fp, fp]
        lib.opt_oracle_rows_round.restype = i32
        _LIB = lib
    return _LIB


def _fp(a):
    assert a.dtype == F and a.flags.c_contiguous
    return a.ctypes.data_as(ctypes.POINTER(ctypes.c_float))


class CShard(object):
    """Same interface as :class:`Shard`, arithmetic done by optimizer_oracle.c."""

    def __init__(self, nelem, opt, hyper=None):
        self.lib = c_lib()
        self.n, self.opt = int(nelem), opt
        self.hyper = tuple(float(F(h)) for h in (hyper or DEFAULT_HYPER[opt]))
        self._hyper = np.array(self.hyper, F)
        self.var = np.zeros(self.n, F)
        self.m, self.v = initial_state(opt, self.hyper, self.n)
        self._step = ctypes.c_int64(0)
        self.scratch = np.zeros(self.n, F)

    @property
    def step(self):
        return self._step.value

    def round(self, slots, mode):
        slots = np.ascontiguousarray(slots, F)
        W, n = slots.shape
        assert n == self.n
        rc = self.lib.opt_oracle_round(self.opt, _fp(self.var), _fp(self.m), _fp(self.v),
                                       _fp(slots), n, W, n, _fp(self._hyper), mode,
                                       _fp(self.scratch), ctypes.byref(self._step))
        assert rc == 0, rc


def c_rows_round(shard, row_len, idx_lists, row_lists, mode):
    """:func:`rows_round` by optimizer_oracle.c on a :class:`CShard`."""
    assert mode in (SUM, SYNC_MEAN)
    W = len(idx_lists)
    idx = [np.ascontiguousarray(i, np.int64) for i in idx_lists]
    rows = [np.ascontiguousarray(r, F).reshape(-1, row_len) for r in row_lists]
    i64p = ctypes.POINTER(ctypes.c_int64)
    fp = ctypes.POINTER(ctypes.c_float)
    pi = (i64p * W)(*[a.ctypes.data_as(i64p) for a in idx])
    pr = (fp * W)(*[a.ctypes.data_as(fp) for a in rows])
    k = (ctypes.c_size_t * W)(*[a.size for a in idx])
    scratch = np.zeros(row_len, F)
    rc = shard.lib.opt_oracle_rows_round(shard.opt, _fp(shard.var), _fp(shard.m), _fp(shard.v),
                                         shard.n // row_len, row_len, W, pi, pr, k,
                                         int(mode == SYNC_MEAN), _fp(shard._hyper), _fp(scratch))
    assert rc == 0, "indices must be strictly ascending and inside the matrix"
    shard._step.value += 1
