"""The Momentum / Adagrad / RMSProp restatements (tests/optimizer_oracle.py and
.c) against each other bit for bit, against hand-computed cases, and the Python
optimizer classes' argument checks."""
import numpy as np
import pytest

from tests import optimizer_oracle as oo
from tfmesos_b200 import engine, psx

F = np.float32
MODES = [oo.ASYNC_ORDERED, oo.SUM, oo.SYNC_MEAN]


def bits(a):
    return np.ascontiguousarray(a, F).view(np.uint32)


def assert_same(a, b, what):
    """Bit-identical, NaN meeting NaN."""
    a, b = np.ascontiguousarray(a, F), np.ascontiguousarray(b, F)
    ok = (bits(a) == bits(b)) | (np.isnan(a) & np.isnan(b))
    assert ok.all(), "%s: %d elements differ" % (what, int((~ok).sum()))


def assert_shards_same(a, b):
    assert_same(a.var, b.var, "var")
    assert_same(a.m, b.m, "m")
    assert_same(a.v, b.v, "v")
    assert a.step == b.step


def test_ids_and_state_counts_match_the_binding():
    assert (oo.MOMENTUM, oo.ADAGRAD, oo.RMSPROP) == (psx.OPT_MOMENTUM, psx.OPT_ADAGRAD,
                                                     psx.OPT_RMSPROP)
    for opt in oo.OPTS:
        assert psx.OPT_STATE_ARRAYS[opt] == oo.STATE_ARRAYS[opt]


@pytest.mark.parametrize("opt", oo.OPTS, ids=lambda o: oo.NAMES[o])
@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("n", [1, 7, 1023, 79510])
def test_numpy_and_c_restatements_agree_bit_for_bit(opt, mode, n):
    rng = np.random.default_rng(n * 10 + opt)
    W = 3
    a, b = oo.Shard(n, opt), oo.CShard(n, opt)
    init = rng.standard_normal(n).astype(F)
    a.var[:] = init
    b.var[:] = init
    for _ in range(4):
        scale = F(10.0 ** rng.integers(-6, 3))
        slots = (rng.standard_normal((W, n)) * scale).astype(F)
        with np.errstate(all="ignore"):
            a.round(slots, mode)
        b.round(slots, mode)
    assert_shards_same(a, b)
    assert a.step == (4 * W if mode == oo.ASYNC_ORDERED else 4)


def _rows_case(rng, n_rows, d):
    """3 workers, overlapping ascending row lists."""
    idx = [np.array([0, 2, 5, n_rows - 1]), np.array([2, 3, 5]), np.array([1, 5, n_rows - 1])]
    rows = [(rng.standard_normal((len(i), d)) * 0.1).astype(F) for i in idx]
    return idx, rows


@pytest.mark.parametrize("opt", oo.OPTS, ids=lambda o: oo.NAMES[o])
@pytest.mark.parametrize("mode", [oo.SUM, oo.SYNC_MEAN])
@pytest.mark.parametrize("d", [200, 7])
def test_rows_round_restatements_agree_and_leave_untouched_rows(opt, mode, d):
    rng = np.random.default_rng(d + opt)
    n_rows = 9
    a, b = oo.Shard(n_rows * d, opt), oo.CShard(n_rows * d, opt)
    init = rng.standard_normal(n_rows * d).astype(F)
    a.var[:] = init
    b.var[:] = init
    m0, v0 = a.m.copy(), a.v.copy()
    for _ in range(2):
        idx, rows = _rows_case(rng, n_rows, d)
        oo.rows_round(a, d, idx, rows, mode)
        oo.c_rows_round(b, d, idx, rows, mode)
    assert_shards_same(a, b)
    assert a.step == 2
    untouched = [4, 6, 7]
    for arr, want in ((a.var, init), (a.m, m0), (a.v, v0)):
        got = arr.reshape(n_rows, d)[untouched]
        assert_same(got, want.reshape(n_rows, d)[untouched], "untouched row")


def _hand(opt, hyper, var, g, steps):
    """Run the numpy and C restatements one slot at a time; return both."""
    shards = [oo.Shard(len(var), opt, hyper), oo.CShard(len(var), opt, hyper)]
    for s in shards:
        s.var[:] = var
        for _ in range(steps):
            s.round(np.asarray(g, F)[None, :], oo.SUM)
    return shards


def test_momentum_hand_case():
    # lr 0.5, mu 0.5, g 1 (binary fractions, exact): a = 1 then 1.5; x = 4 - .5 - .75
    for s in _hand(oo.MOMENTUM, (0.5, 0.5, 0, 0), [4.0], [1.0], 2):
        assert s.m[0] == F(1.5) and s.var[0] == F(2.75)


def test_adagrad_hand_case():
    # init 3, g 1: a = 4, x = 1 - (1 * 0.5) * (1 / 2) = 0.75; again: a = 5
    for s in _hand(oo.ADAGRAD, (0.5, 3.0, 0, 0), [1.0], [1.0], 1):
        assert s.m[0] == F(4.0) and s.var[0] == F(0.75)
    for s in _hand(oo.ADAGRAD, (0.5, 3.0, 0, 0), [1.0], [1.0], 2):
        want = F(F(0.75) - F(F(0.5) * F(F(1) / np.sqrt(F(5)))))
        assert s.m[0] == F(5.0) and s.var[0] == want


def test_rmsprop_hand_case():
    # decay 0.75, mu 0.5, eps 0, lr 1, g 2: ms = 1 + (4 - 1) * 0.25 = 1.75;
    # mom = 0 * 0.5 + 2 / sqrt(1.75); x = 3 - mom
    for s in _hand(oo.RMSPROP, (1.0, 0.75, 0.5, 0.0), [3.0], [2.0], 1):
        mom = F(F(2) / np.sqrt(F(1.75)))
        assert s.m[0] == F(1.75) and s.v[0] == mom and s.var[0] == F(F(3) - mom)


def test_initial_state_is_tf_slot_initialisation():
    assert (oo.Shard(3, oo.MOMENTUM).m == 0).all()
    assert (oo.Shard(3, oo.ADAGRAD, (0.1, 0.25, 0, 0)).m == F(0.25)).all()
    s = oo.Shard(3, oo.RMSPROP)
    assert (s.m == 1).all() and (s.v == 0).all()


@pytest.mark.parametrize("bad", [0.0, -0.1, float("nan")])
def test_adagrad_rejects_non_positive_initial_accumulator(bad):
    with pytest.raises(ValueError, match="initial_accumulator_value"):
        engine.AdagradOptimizer(0.1, initial_accumulator_value=bad)


def test_optimizer_classes_carry_tf_defaults_and_the_header_tuple():
    from tfmesos_b200 import train
    assert engine.GradientDescentOptimizer(0.5).hyper == (0.5, 0.9, 0.999, 1e-8)
    assert engine.AdamOptimizer(0.01).hyper == (0.01, 0.9, 0.999, 1e-8)
    m = train.MomentumOptimizer(2.0, 0.9)
    assert (m.opt, m.hyper) == (psx.OPT_MOMENTUM, (2.0, 0.9, 0.0, 0.0))
    a = train.AdagradOptimizer(3.0)
    assert (a.opt, a.hyper) == (psx.OPT_ADAGRAD, (3.0, 0.1, 0.0, 0.0))
    r = train.RMSPropOptimizer(0.01)
    assert (r.opt, r.hyper) == (psx.OPT_RMSPROP, (0.01, 0.9, 0.0, 1e-10))
