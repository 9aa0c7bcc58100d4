"""Momentum, Adagrad and RMSProp through libpsx.so on one GPU, against the C
restatement (tests/optimizer_oracle.c) bit for bit: var, the state arrays and
global_step, on every path the kernels serve -- the staged apply, the fused
psx_round, the served loop, index-list rows, the BASELINE-size buckets,
checkpoints and the ParameterClient session."""
import numpy as np
import pytest

from oracle import ps_oracle as o
from tests import optimizer_oracle as oo
from tfmesos_b200 import checkpoint, engine, psx

pytestmark = pytest.mark.gpu
F = np.float32
MODES = [psx.MODE_ASYNC_ORDERED, psx.MODE_SUM, psx.MODE_SYNC_MEAN]
OPTS = list(oo.OPTS)
OPT_IDS = [oo.NAMES[x] for x in OPTS]
RESNET50_BUCKET = 25_557_032
NMF_W = 200_000_000


@pytest.fixture(scope="module", autouse=True)
def _init():
    import torch
    assert torch.cuda.is_available(), "gpu tests need a CUDA device"
    psx.init(0)
    yield
    torch.cuda.synchronize()


def bits(a):
    return np.ascontiguousarray(a, F).view(np.uint32)


def assert_bits_equal(got, want, what):
    """Same bits everywhere; a NaN must meet a NaN."""
    g, w = bits(got).ravel(), bits(want).ravel()
    both_nan = np.isnan(np.ascontiguousarray(got, F).ravel()) & \
        np.isnan(np.ascontiguousarray(want, F).ravel())
    bad = np.nonzero((g != w) & ~both_nan)[0]
    assert bad.size == 0, "%s: %d of %d elements differ, first at %d: got %r want %r" % (
        what, bad.size, g.size, bad[0], got.ravel()[bad[0]], want.ravel()[bad[0]])


def make_optimizer(opt, hyper):
    if opt == oo.MOMENTUM:
        return engine.MomentumOptimizer(hyper[0], hyper[1])
    if opt == oo.ADAGRAD:
        return engine.AdagradOptimizer(hyper[0], hyper[1])
    return engine.RMSPropOptimizer(*hyper)


def check_shard(shard, ref, what=""):
    assert_bits_equal(shard.get_values(psx.VAR), ref.var, what + " var")
    assert_bits_equal(shard.get_values(psx.M), ref.m, what + " m")
    if oo.STATE_ARRAYS[ref.opt] == 2:
        assert_bits_equal(shard.get_values(psx.V), ref.v, what + " v")
    st = shard.state()
    assert st["global_step"] == ref.step
    # no beta powers: the stored values stay what creation put there
    assert (F(st["beta1_power"]), F(st["beta2_power"])) == (F(ref.hyper[1]), F(ref.hyper[2]))


def run_rounds(n, opt, mode, W, rounds, wire=psx.F32, seed=0, hyper=None):
    import torch
    rng = np.random.default_rng(seed)
    ref = oo.CShard(n, opt, hyper)
    shard = psx.Shard(0, n, opt, *ref.hyper, n_slots=W, wire=wire)
    init = rng.standard_normal(n).astype(F)
    shard.set_values(psx.VAR, init)
    ref.var[:] = init
    clients = [psx.Client(shard.export(), 0, w) for w in range(W)]
    try:
        for r in range(rounds):
            scale = F(10.0 ** rng.integers(-5, 3))
            slots = (rng.standard_normal((W, n)) * scale).astype(F)
            dev = torch.from_numpy(slots).cuda()
            for w in range(W):
                clients[w].push(dev[w].data_ptr(), n, seq=r + 1)
            shard.apply(mode, 0, W, wait_seq=r + 1)
            if wire == psx.BF16:
                slots = o.bf16_to_f32(o.f32_to_bf16(slots)).reshape(W, n)
            ref.round(slots, mode)
            del dev
        torch.cuda.synchronize()
        return shard, ref, clients
    except Exception:
        for c in clients:
            c.close()
        shard.destroy()
        raise


def close(shard, clients):
    for c in clients:
        c.close()
    shard.destroy()


# ------------------------------------------------------------ staged apply ----
@pytest.mark.parametrize("opt", OPTS, ids=OPT_IDS)
@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("wire", [psx.F32, psx.BF16], ids=["f32", "bf16"])
@pytest.mark.parametrize("n,W", [(1, 1), (7, 3), (1023, 2), (7850, 2), (79510, 5),
                                 (400000, 4), (1 << 20, 2)])
def test_apply_bit_exact_vs_oracle(opt, mode, wire, n, W):
    shard, ref, clients = run_rounds(n, opt, mode, W, rounds=4, wire=wire, seed=n + W + opt)
    try:
        check_shard(shard, ref)
        assert shard.state()["apply_seq"] == 4
    finally:
        close(shard, clients)


@pytest.mark.parametrize("opt", OPTS, ids=OPT_IDS)
def test_fresh_shard_holds_tf_initial_state(opt):
    hyper = (0.5, 0.25, 0.5, 1e-3)
    shard = psx.Shard(0, 5000, opt, *hyper, n_slots=1)
    try:
        m0, v0 = oo.initial_state(opt, hyper, 5000)
        assert_bits_equal(shard.get_values(psx.M), m0, "m")
        if oo.STATE_ARRAYS[opt] == 2:
            assert_bits_equal(shard.get_values(psx.V), v0, "v")
        else:
            with pytest.raises(RuntimeError, match="no region"):
                shard.get_values(psx.V)
    finally:
        shard.destroy()


def test_creation_errors():
    with pytest.raises(RuntimeError, match="unknown optimizer"):
        psx.Shard(0, 100, 5, n_slots=1)
    with pytest.raises(RuntimeError, match="unknown optimizer"):
        psx.Shard(0, 100, -1, n_slots=1)
    for bad in (0.0, -0.5, float("nan")):
        with pytest.raises(RuntimeError, match="initial_accumulator_value"):
            psx.Shard(0, 100, psx.OPT_ADAGRAD, 0.1, bad, 0.0, 0.0, n_slots=1)


# -------------------------------------------------------------- fused round ----
@pytest.mark.parametrize("opt", OPTS, ids=OPT_IDS)
@pytest.mark.parametrize("mode", MODES)
def test_fused_round_bit_exact_and_scatters_parameters(opt, mode):
    import torch
    W = 3
    rng = np.random.default_rng(7 + opt)
    variables = [("hid_w", (784, 100)), ("hid_b", (100,)), ("sm_w", (100, 10)), ("sm_b", (10,))]
    hyper = oo.DEFAULT_HYPER[opt]
    cl = engine.LocalCluster(variables, 1, W, make_optimizer(opt, hyper), fused=True)
    nb = cl.layout.bucket_nelem[0]
    ref = oo.CShard(nb, opt, hyper)
    try:
        init = rng.standard_normal(nb).astype(F)
        cl.servers[(0, 0)].shard.set_values(psx.VAR, init)
        ref.var[:] = init
        for r in range(3):
            slots = (rng.standard_normal((W, nb)) * 0.1).astype(F)
            for w in range(W):
                cl.workers[w].grad_flat[0][:nb].copy_(torch.from_numpy(slots[w]))
            cl.round(mode)
            ref.round(slots, mode)
        torch.cuda.synchronize()
        check_shard(cl.servers[(0, 0)].shard, ref)
        for w in range(W):
            assert_bits_equal(cl.workers[w].param_flat[0][:nb].cpu().numpy(), ref.var,
                              "worker %d params" % w)
        assert cl.global_step() == ref.step
    finally:
        cl.close()


# ------------------------------------------------------------ served loop ----
N_SERVE = 79510


def _grad(w, r, n=N_SERVE):
    return (np.random.default_rng(100 * w + r).standard_normal(n) * 0.1).astype(F)


class _Rig(object):
    """W in-process workers on one served shard (workers wait on the host)."""

    def __init__(self, W, opt, hyper, wire=psx.F32):
        import torch
        self.torch, self.W, self.n = torch, W, N_SERVE
        self.ref = oo.CShard(self.n, opt, hyper)
        self.shard = psx.Shard(0, self.n, opt, *self.ref.hyper, n_slots=W, wire=wire)
        init = np.random.default_rng(5).standard_normal(self.n).astype(F)
        self.shard.set_values(psx.VAR, init)
        self.ref.var[:] = init
        self.clients = [psx.Client(self.shard.export(), 0, w) for w in range(W)]
        for w, c in enumerate(self.clients):
            self.shard.register_client(w, c.export())
        self.streams = [torch.cuda.Stream(device=0) for _ in range(W)]
        self.grads = [torch.zeros(self.n, device="cuda") for _ in range(W)]
        self.params = [torch.zeros(self.n, device="cuda") for _ in range(W)]

    def push(self, w, seq, g, stamp=0):
        with self.torch.cuda.stream(self.streams[w]):
            self.grads[w].copy_(self.torch.from_numpy(g), non_blocking=False)
        self.clients[w].push_stamped(self.grads[w].data_ptr(), self.n, 0, psx.F32, seq, stamp,
                                     self.streams[w])

    def close(self):
        self.shard.serve_stop()
        for w, c in enumerate(self.clients):
            self.shard.unregister_client(w)
            c.close()
        self.shard.destroy()


@pytest.mark.parametrize("opt", OPTS, ids=OPT_IDS)
def test_served_async_fixed_arrival_order_bit_exact(opt):
    rig = _Rig(3, opt, oo.DEFAULT_HYPER[opt])
    try:
        rig.shard.serve_start(psx.MODE_ASYNC_ORDERED)
        seqs = [0, 0, 0]
        for k, w in enumerate([2, 0, 1, 1, 2, 0, 0, 2, 1]):
            seqs[w] += 1
            g = _grad(w, seqs[w])
            rig.push(w, seqs[w], g)
            c, st = rig.clients[w], rig.streams[w]
            st.synchronize()
            c.wait_host("applied", seqs[w])
            c.pull(rig.params[w].data_ptr(), rig.n, 0, psx.F32, 0, st)
            st.synchronize()
            rig.ref.round(g[None, :], oo.ASYNC_ORDERED)
            assert_bits_equal(rig.params[w].cpu().numpy(), rig.ref.var, "pull %d" % k)
        check_shard(rig.shard, rig.ref)
    finally:
        rig.close()


@pytest.mark.parametrize("opt", OPTS, ids=OPT_IDS)
def test_served_sync_mean_all_replicas_bit_exact(opt):
    W = 3
    rig = _Rig(W, opt, oo.DEFAULT_HYPER[opt])
    try:
        rig.shard.serve_start(psx.MODE_SYNC_MEAN, replicas_to_aggregate=W)
        for r in range(1, 4):
            slots = []
            for w in range(W):
                g = _grad(w, r)
                rig.push(w, r, g, stamp=r - 1)
                slots.append(g)
            for w in range(W):
                rig.streams[w].synchronize()
                rig.clients[w].wait_host("tokens", r)
            rig.ref.round(np.stack(slots), oo.SYNC_MEAN)
        check_shard(rig.shard, rig.ref)
        assert rig.shard.serve_stats()["dropped"] == 0
    finally:
        rig.close()


# --------------------------------------------------------------------- rows ----
@pytest.mark.parametrize("opt", OPTS, ids=OPT_IDS)
@pytest.mark.parametrize("mode", [psx.MODE_SUM, psx.MODE_SYNC_MEAN])
@pytest.mark.parametrize("d", [200, 7])
def test_rows_from_three_workers_with_overlaps_bit_exact(opt, mode, d):
    import torch
    n_rows, W, R = 4096, 3, 3
    ref = oo.CShard(n_rows * d, opt)
    shard = psx.Shard(0, n_rows * d, opt, *ref.hyper, n_slots=W)
    init = np.random.default_rng(11).standard_normal(n_rows * d).astype(F)
    shard.set_values(psx.VAR, init)
    ref.var[:] = init
    clients = [psx.Client(shard.export(), 0, w) for w in range(W)]
    rng = np.random.default_rng(d + opt)
    touched = np.zeros(n_rows, bool)
    try:
        for r in range(1, R + 1):
            idx_lists, row_lists, keep = [], [], []
            for w in range(W):
                k = int(rng.integers(1, 900))
                idx = np.sort(rng.choice(n_rows, size=k, replace=False)).astype(np.int64)
                if w == 2:
                    idx = np.unique(np.concatenate([idx, idx_lists[0][:50], idx_lists[1][-30:]]))
                rows = (rng.standard_normal((idx.size, d)) * 0.1).astype(F)
                idx_lists.append(idx)
                row_lists.append(rows)
                touched[idx] = True
                ti, tr = torch.from_numpy(idx).cuda(), torch.from_numpy(rows).cuda()
                keep.append((ti, tr))
                clients[w].push_rows(ti.data_ptr(), tr.data_ptr(), idx.size, d, psx.F32, r)
            shard.apply_rows(mode, 0, W, d, wait_seq=r)
            torch.cuda.synchronize()
            oo.c_rows_round(ref, d, idx_lists, row_lists, mode)
        check_shard(shard, ref)
        # lazy: untouched rows keep var and state exactly
        m0, v0 = oo.initial_state(opt, ref.hyper, n_rows * d)
        un = ~touched
        assert un.any()
        assert_bits_equal(shard.get_values(psx.VAR).reshape(n_rows, d)[un],
                          init.reshape(n_rows, d)[un], "untouched var")
        assert_bits_equal(shard.get_values(psx.M).reshape(n_rows, d)[un],
                          m0.reshape(n_rows, d)[un], "untouched m")
    finally:
        close(shard, clients)


# ---------------------------------------------------------- BASELINE sizes ----
@pytest.mark.parametrize("opt", OPTS, ids=OPT_IDS)
def test_resnet50_bucket_bf16_async_bit_exact(opt):
    shard, ref, clients = run_rounds(RESNET50_BUCKET, opt, psx.MODE_ASYNC_ORDERED, 2, rounds=2,
                                     wire=psx.BF16, seed=50 + opt)
    try:
        check_shard(shard, ref, "resnet50")
    finally:
        close(shard, clients)


def test_nmf_2e8_momentum_bit_exact():
    shard, ref, clients = run_rounds(NMF_W, oo.MOMENTUM, psx.MODE_SUM, 1, rounds=2, seed=2)
    try:
        check_shard(shard, ref, "nmf")
    finally:
        close(shard, clients)


# ------------------------------------------------------------- checkpoints ----
VARS = [("hid_w", (784, 100)), ("hid_b", (100,)), ("sm_w", (100, 10)), ("sm_b", (10,))]


def _rounds(cl, rng, k):
    import torch
    for _ in range(k):
        for w in cl.workers:
            for name, (task, off, shape, numel) in cl.layout.entries.items():
                w.grads[name].copy_(torch.from_numpy(
                    (rng.standard_normal(numel) * 0.1).astype(F)).view(shape))
        cl.round(psx.MODE_ASYNC_ORDERED)
    torch.cuda.synchronize()


def _snapshot(cl, opt):
    out = {}
    for key, ps in cl.servers.items():
        regions = [psx.VAR, psx.M, psx.V][:1 + oo.STATE_ARRAYS[opt]]
        out[key] = ([ps.shard.get_values(r) for r in regions], ps.shard.state())
    return out


@pytest.mark.parametrize("opt", [oo.MOMENTUM, oo.RMSPROP], ids=["momentum", "rmsprop"])
def test_checkpoint_resume_is_bit_identical(tmp_path, opt):
    hyper = oo.DEFAULT_HYPER[opt]
    a = engine.LocalCluster(VARS, 2, 2, make_optimizer(opt, hyper))
    try:
        a.set_variable("hid_w", np.random.default_rng(1).standard_normal((784, 100)).astype(F))
        _rounds(a, np.random.default_rng(5), 3)
        path = str(tmp_path / "ckpt")
        checkpoint.save(a, path)
        _rounds(a, np.random.default_rng(6), 2)
        want = _snapshot(a, opt)
    finally:
        a.close()
    b = engine.LocalCluster(VARS, 2, 2, make_optimizer(opt, hyper))
    try:
        checkpoint.restore(b, path)
        assert b.global_step() == 6
        for w in b.workers:
            w.pull()
        _rounds(b, np.random.default_rng(6), 2)
        got = _snapshot(b, opt)
    finally:
        b.close()
    assert sorted(got) == sorted(want)
    for key in want:
        for i, (g, w) in enumerate(zip(got[key][0], want[key][0])):
            assert_bits_equal(g, w, "%r region %d" % (key, i))
        assert got[key][1]["global_step"] == want[key][1]["global_step"] == 10
    # a checkpoint of one optimizer does not restore into another
    c = engine.LocalCluster(VARS, 2, 2, engine.AdamOptimizer(0.01))
    try:
        with pytest.raises(RuntimeError, match="does not match"):
            checkpoint.restore(c, path)
    finally:
        c.close()


# ------------------------------------------------------ ParameterClient ----
def test_parameter_client_momentum_bit_exact(tmp_path):
    import socket
    import threading

    from tfmesos_b200 import train as tf

    socks = [socket.socket() for _ in range(1)]
    for s in socks:
        s.bind(("127.0.0.1", 0))
    port = socks[0].getsockname()[1]
    for s in socks:
        s.close()
    spec = {"ps": ["127.0.0.1:%d" % port], "worker": ["127.0.0.1:1"]}
    server = tf.Server(spec, "ps", 0)
    t = threading.Thread(target=server.join)
    t.daemon = True
    t.start()
    hyper = (0.05, 0.9, 0.0, 0.0)
    variables = [("w", (300, 20)), ("b", (20,))]
    rng = np.random.default_rng(21)
    init = {"w": rng.standard_normal((300, 20)).astype(F), "b": rng.standard_normal(20).astype(F)}
    refs = {k: oo.CShard(v.size, oo.MOMENTUM, hyper) for k, v in init.items()}
    for k, v in init.items():
        refs[k].var[:] = v.ravel()
    try:
        sess = tf.ParameterClient(spec, variables, tf.MomentumOptimizer(hyper[0], hyper[1]), 0,
                                  device=0, init=init)
        import torch
        for _ in range(4):
            for k, v in init.items():
                g = (rng.standard_normal(v.shape) * 0.1).astype(F)
                sess.grads[k].copy_(torch.from_numpy(g))
                refs[k].round(g.reshape(1, -1), oo.ASYNC_ORDERED)
            step = sess.minimize()
        assert step == 4
        for k in init:
            assert_bits_equal(sess.read(k).ravel(), refs[k].var, k)
            assert_bits_equal(sess.params[k].cpu().numpy().ravel(), refs[k].var, k + " pulled")
        sess.close()
    finally:
        server.endpoint.stop_event.set()
