"""The learning-rate schedules ExponentialDecay, InverseTimeDecay, PolynomialDecay and PiecewiseConstantDecay on the
device, against the oracle (tests/schedule_oracle.py on tests/optimizer_oracle.py) with the bars of
tests/test_gpu_optimizers.py: every fit kernel, both unit-split builds, many-model, weighted and ragged launches, the
LSTM kernel, the boundary of a piecewise schedule to the bit, the schedule across fit calls and from a set
`iterations`, the batched surface and the plugins end to end."""
import logging

import numpy as np
import pytest

from oracle import keras_lstm as kl, keras_mlp as km
import optimizer_oracle as oo
import schedule_oracle as so
import weighted_oracle as wo
from helpers import lstm_factory, lstm_sequences, synthetic_targets
from bore_b200 import layers
from bore_b200.schedules import ExponentialDecay, InverseTimeDecay, PiecewiseConstantDecay, PolynomialDecay

pytestmark = pytest.mark.gpu

LOSS_TOL = 1e-4

# decay_steps of 10 to 40 in fits of about 70 steps: the rate changes materially within the run
SCHEDULES = {
    "exponential": lambda s=1.0: ExponentialDecay(1e-2 * s, 20, 0.5),
    "exponential_staircase": lambda s=1.0: ExponentialDecay(1e-2 * s, 15, 0.5, staircase=True),
    "inverse_time": lambda s=1.0: InverseTimeDecay(1e-2 * s, 10, 1.0),
    "inverse_time_staircase": lambda s=1.0: InverseTimeDecay(1e-2 * s, 12, 1.0, staircase=True),
    "polynomial": lambda s=1.0: PolynomialDecay(1e-2 * s, 40, 1e-3 * s, power=2.0),
    "polynomial_cycle": lambda s=1.0: PolynomialDecay(1e-2 * s, 25, 1e-3 * s, cycle=True),
    "piecewise": lambda s=1.0: PiecewiseConstantDecay([18, 36, 54], [1e-2 * s, 5e-3 * s, 2e-3 * s, 1e-3 * s]),
}
KINDS = {
    "adam": lambda lr: layers.Adam(learning_rate=lr),
    "rmsprop_momentum": lambda lr: layers.RMSprop(learning_rate=lr, momentum=0.9),
    "adagrad": lambda lr: layers.Adagrad(learning_rate=lr),
    "rmsprop": lambda lr: layers.RMSprop(learning_rate=lr),
    "adadelta": lambda lr: layers.Adadelta(learning_rate=lr),
    "adamax": lambda lr: layers.Adamax(learning_rate=lr),
}


@pytest.fixture(autouse=True, scope="module")
def _optimizer_oracle():
    with oo.installed():
        yield


def make(kind, sched, scale=1.0):
    return KINDS[kind](SCHEDULES[sched](100.0 if kind == "adadelta" else scale))


def _problem(dims, N, E, seed):
    rs = np.random.RandomState(seed)
    X = rs.uniform(size=(N, dims[0]))
    y = synthetic_targets(X)
    return X, y < np.quantile(y, 0.25), np.stack([rs.permutation(N) for _ in range(E)])


def _net(dims, acts, o, w=None, n_models=1):
    from bore_b200.engine import NativeMLP
    net = NativeMLP(dims, acts, n_models=n_models)
    net.set_optimizer_kind(o)
    if w is not None:
        for i in range(n_models):
            net.set_weights(w, model=i)
    return net


def _oracle_fit(w0, acts, X, z, E, perms, o, l2=0.0, st=None):
    w = [a.copy() for a in w0]
    st = oo.state_for(w, o) if st is None else st
    with so.installed(o.learning_rate):
        h, st = km.fit(w, acts, X, z, E, 64, perms, adam=st, l2=l2)
    return h, w, st


def _close(net, h, w_ref, h_ref, model=0):
    assert np.abs(np.asarray(h) - h_ref).max() <= LOSS_TOL, np.abs(np.asarray(h) - h_ref).max()
    for a, b in zip(net.get_weights(model=model), w_ref):
        assert np.abs(a - b).max() <= 2e-3


DIMS, ACTS = [6, 32, 32, 1], ["elu", "elu", "sigmoid"]


@pytest.mark.parametrize("mode", [1, 2, 3, 4])
@pytest.mark.parametrize("sched", sorted(SCHEDULES))
@pytest.mark.parametrize("kind", ["adam", "rmsprop_momentum", "adagrad"])
@pytest.mark.parametrize("l2", [0.0, 1e-3])
def test_fit_modes(mode, sched, kind, l2):
    o = make(kind, sched)
    N, E = 333, 12  # 72 steps
    X, z, perms = _problem(DIMS, N, E, seed=5)
    w0 = km.init_weights(DIMS, 3)
    h_ref, w_ref, st = _oracle_fit(w0, ACTS, X, z, E, perms, o, l2)
    net = _net(DIMS, ACTS, o, w0)
    net.set_fit_mode(mode)
    _close(net, net.fit(X, z, E, 64, perms, l2=l2), w_ref, h_ref)
    assert net.get_optimizer_state()[2] == st.t == E * 6


@pytest.mark.parametrize("mode", [1, 4])
@pytest.mark.parametrize("kind", ["rmsprop", "adadelta", "adamax"])
def test_other_kinds(mode, kind):
    o = make(kind, "inverse_time")
    N, E = 333, 12
    X, z, perms = _problem(DIMS, N, E, seed=6)
    w0 = km.init_weights(DIMS, 4)
    h_ref, w_ref, _ = _oracle_fit(w0, ACTS, X, z, E, perms, o)
    net = _net(DIMS, ACTS, o, w0)
    net.set_fit_mode(mode)
    _close(net, net.fit(X, z, E, 64, perms), w_ref, h_ref)


@pytest.mark.parametrize("dims", [[50, 64, 64, 64, 1], [6, 32, 32, 1], [6, 16, 16, 1], [7, 24, 24, 1],
                                  [7, 40, 40, 1]])
@pytest.mark.parametrize("kind,sched", [("adam", "exponential"), ("rmsprop_momentum", "piecewise"),
                                        ("adagrad", "polynomial_cycle")])
def test_unit_split_builds(dims, kind, sched):
    """Fit mode 4: hidden widths 16 / 32 / 64 take the compile-time builds of the unit-split kernel, 24 / 40 its
    run-time build."""
    o = make(kind, sched)
    acts = ["tanh"] * (len(dims) - 2) + ["sigmoid"]
    N, E = 700, 6  # 66 steps
    X, z, perms = _problem(dims, N, E, seed=9)
    w0 = km.init_weights(dims, 4)
    h_ref, w_ref, _ = _oracle_fit(w0, acts, X, z, E, perms, o)
    net = _net(dims, acts, o, w0)
    net.set_fit_mode(4)
    _close(net, net.fit(X, z, E, 64, perms), w_ref, h_ref)


@pytest.mark.parametrize("M", [20, 600])
@pytest.mark.parametrize("kind,sched", [("adam", "exponential_staircase"), ("adamax", "polynomial"),
                                        ("adadelta", "piecewise")])
def test_many_models(M, kind, sched):
    o = make(kind, sched)
    N, E = 150, 24  # 72 steps
    probs = [_problem(DIMS, N, E, seed=50 + i) for i in range(M)]
    ws = [km.init_weights(DIMS, 200 + i) for i in range(M)]
    net = _net(DIMS, ACTS, o, n_models=M)
    for i, w in enumerate(ws):
        net.set_weights(w, model=i)
    Xd = net.to_device(np.concatenate([p[0] for p in probs]), np.float32)
    zd = net.to_device(np.concatenate([p[1] for p in probs]).astype(np.float32), np.float32)
    pd = net.to_device(np.stack([p[2] for p in probs]).astype(np.int32), np.int32)
    loss = net.fit_dev(Xd, zd, N, 64, E, pd, model0=0, count=M, shared_data=False, shared_perm=False).cpu().numpy()
    for i in list(range(0, M, max(1, M // 25))) + [M - 1]:
        h_ref, _, _ = _oracle_fit(ws[i], ACTS, probs[i][0], probs[i][1], E, probs[i][2], o)
        assert np.abs(loss[i] - h_ref).max() <= LOSS_TOL, i


@pytest.mark.parametrize("kind,sched", [("adam", "piecewise"), ("rmsprop_momentum", "exponential")])
def test_weighted_fit(kind, sched):
    o = make(kind, sched)
    N, E = 200, 18  # 72 steps
    X, z, perms = _problem(DIMS, N, E, seed=11)
    sw = np.random.RandomState(12).uniform(0, 2, size=N).astype(np.float32)
    w0 = km.init_weights(DIMS, 6)
    w_ref = [a.copy() for a in w0]
    with so.installed(o.learning_rate):
        h_ref, _ = wo.fit(w_ref, ACTS, X, z, E, 64, perms, sample_weight=sw, class_weight={0: 0.5, 1: 2.0},
                          adam=oo.state_for(w_ref, o))
    for mode in (1, 2, 4):
        net = _net(DIMS, ACTS, o, w0)
        net.set_fit_mode(mode)
        _close(net, net.fit(X, z, E, 64, perms, w=sw, class_weight=(0.5, 2.0)), w_ref, h_ref)


@pytest.mark.parametrize("kind,sched", [("adam", "inverse_time_staircase"), ("adagrad", "piecewise")])
def test_ragged_fit(kind, sched):
    """Problems with other epoch counts: each model's own `iterations` drives its schedule."""
    from bore_b200.ragged import RaggedLayout
    o = make(kind, sched)
    n, e = np.array([40, 130, 75]), np.array([40, 24, 30])
    lay = RaggedLayout(n, e)
    probs = [_problem(DIMS, int(n[p]), int(e[p]), seed=20 + p) for p in range(3)]
    ws = [km.init_weights(DIMS, 30 + p) for p in range(3)]
    net = _net(DIMS, ACTS, o, n_models=3)
    for p, w in enumerate(ws):
        net.set_weights(w, model=p)
    Xd = net.to_device(np.concatenate([p[0] for p in probs]), np.float32)
    zd = net.to_device(np.concatenate([p[1] for p in probs]).astype(np.float32), np.float32)
    pd = net.to_device(np.concatenate([p[2].reshape(-1) for p in probs]).astype(np.int32), np.int32)
    loss = net.fit_ragged_dev(Xd, zd, lay, 64, pd).cpu().numpy()
    for p in range(3):
        h_ref, w_ref, st = _oracle_fit(ws[p], ACTS, probs[p][0], probs[p][1], int(e[p]), probs[p][2], o)
        _close(net, loss[lay.losses[p]:lay.losses[p + 1]], w_ref, h_ref, model=p)
        assert net.get_optimizer_state(model=p)[2] == st.t


@pytest.mark.parametrize("mode", [0, 1, 4])
def test_two_fits_follow_one_oracle_run(mode):
    o = make("adam", "piecewise")
    N, E = 200, 18
    X, z, perms = _problem(DIMS, N, E, seed=14)
    w0 = km.init_weights(DIMS, 8)
    h_ref, w_ref, _ = _oracle_fit(w0, ACTS, X, z, E, perms, o)
    net = _net(DIMS, ACTS, o, w0)
    net.set_fit_mode(mode)
    ha = net.fit(X, z, 7, 64, perms[:7])
    hb = net.fit(X, z, E - 7, 64, perms[7:])
    _close(net, np.concatenate([ha, hb]), w_ref, h_ref)


@pytest.mark.parametrize("kind", ["adam", "adagrad"])
def test_schedule_starts_at_the_set_iterations(kind):
    """set_optimizer_state(..., iterations=k): update t of the next fit takes the schedule at k + t - 1."""
    o = make(kind, "exponential")
    k, N, E = 40, 200, 6
    X, z, perms = _problem(DIMS, N, E, seed=15)
    w0 = km.init_weights(DIMS, 9)
    w = [a.copy() for a in w0]
    st = oo.state_for(w, o)
    st.t = k
    h_ref, w_ref, st = _oracle_fit(w0, ACTS, X, z, E, perms, o, st=st)
    net = _net(DIMS, ACTS, o, w0)
    s0, s1, _ = net.get_optimizer_state()
    net.set_optimizer_state(s0, s1, k)
    _close(net, net.fit(X, z, E, 64, perms), w_ref, h_ref)
    assert net.get_optimizer_state()[2] == st.t == k + E * 4
    # the same fit from iterations = 0 ends elsewhere: the schedule did start at k
    fresh = _net(DIMS, ACTS, o, w0)
    fresh.fit(X, z, E, 64, perms)
    assert max(np.abs(a - b).max() for a, b in zip(fresh.get_weights(), w_ref)) > 1e-3


def test_new_schedule_keeps_the_state():
    o = make("adagrad", "exponential")
    N, E = 200, 4
    X, z, perms = _problem(DIMS, N, E, seed=16)
    net = _net(DIMS, ACTS, o, km.init_weights(DIMS, 10))
    net.fit(X, z, E, 64, perms)
    before = net.get_optimizer_state()
    net.set_optimizer_kind(make("adagrad", "piecewise"))
    after = net.get_optimizer_state()
    assert after[2] == before[2] == E * 4
    assert all(np.array_equal(a, b) for a, b in zip(before[0], after[0]))
    net.set_optimizer_kind(layers.Adagrad(learning_rate=1e-2))  # back to a constant rate: the same build rule
    assert net.get_optimizer_state()[2] == E * 4


# ---------------------------------------------------------------------------------------------- boundaries, to the bit
def _piecewise(b, lo, hi, kind="adam"):
    return KINDS[kind](PiecewiseConstantDecay([b], [lo, hi]))


@pytest.mark.parametrize("mode,dims", [(1, [6, 32, 32, 1]), (4, [6, 32, 32, 1]), (4, [7, 24, 24, 1])])
@pytest.mark.parametrize("kind", ["adam", "adagrad"])
def test_boundary_placement_mlp(mode, dims, kind):
    """Update t takes the schedule at t - 1: with the boundary at b = E1 * steps_per_epoch - 1, the first E1
    epochs run at the rate of values[0] and every later update at values[1].  Under Adam and Adagrad an update at
    rate 0 leaves a parameter exactly where it was (RMSprop's momentum would still move it)."""
    acts = ["elu"] * (len(dims) - 2) + ["sigmoid"]
    N, E1, E2, lr = 128, 5, 9, 1e-2
    spe = 2
    b = E1 * spe - 1
    X, z, perms = _problem(dims, N, E2, seed=17)
    w0 = km.init_weights(dims, 11)

    def run(o, E):
        net = _net(dims, acts, o, w0)
        net.set_fit_mode(mode)
        net.fit(X, z, E, 64, perms[:E])
        return net.get_weights()

    stop = run(_piecewise(b, lr, 0.0, kind), E2)  # rate 0 from update b + 2 on: an update leaves w exactly
    short = run(_piecewise(b, lr, lr, kind), E1)
    assert all(np.array_equal(a, c) for a, c in zip(stop, short))
    assert max(np.abs(a - c).max() for a, c in zip(short, w0)) > 1e-3
    late = run(_piecewise(b, 0.0, lr, kind), E1)  # rate 0 for updates 1 .. b + 1
    assert all(np.array_equal(a, np.asarray(c, np.float32)) for a, c in zip(late, w0))
    moved = run(_piecewise(b, 0.0, lr, kind), E1 + 1)
    assert max(np.abs(a - c).max() for a, c in zip(moved, w0)) > 1e-4


def _lstm(D, U, L, o, w0, mv):
    from bore_b200.layers import BinaryCrossentropy
    net = lstm_factory(D, U, L, "tanh").build_many_to_many(mask_value=mv)
    net.compile(optimizer=o, loss=BinaryCrossentropy(from_logits=True))
    net.set_weights(w0)
    return net


@pytest.mark.parametrize("kind", ["adam", "adagrad"])
def test_boundary_placement_lstm(kind):
    D, U, L, N, B, T, mv = 8, 32, 2, 100, 50, 4, -1.0
    E1, E2, lr = 3, 6, 1e-2
    b = E1 * 2 - 1
    X, Y = lstm_sequences(4, N, T, D, mv)
    rs = np.random.RandomState(5)
    perms = np.stack([rs.permutation(N) for _ in range(E2)])
    w0 = kl.init_weights(D, U, L, seed=6)

    def run(o, E):
        net = _lstm(D, U, L, o, w0, mv)
        net.fit(X, Y, epochs=E, batch_size=B, permutations=perms[:E], verbose=0)
        return net.get_weights()

    stop, short = run(_piecewise(b, lr, 0.0, kind), E2), run(_piecewise(b, lr, lr, kind), E1)
    assert all(np.array_equal(a, c) for a, c in zip(stop, short))
    assert max(np.abs(a - c).max() for a, c in zip(short, w0)) > 1e-3
    late = run(_piecewise(b, 0.0, lr, kind), E1)
    assert all(np.array_equal(a, np.asarray(c, np.float32)) for a, c in zip(late, w0))


# ---------------------------------------------------------------------------------------------- LSTM
@pytest.mark.parametrize("sched", sorted(SCHEDULES))
@pytest.mark.parametrize("kind", ["adam", "rmsprop_momentum", "adagrad"])
def test_lstm(sched, kind):
    """The LSTM fit kernel against keras_lstm with the bars of tests/test_gpu_lstm.py; two fit calls continue the
    schedule of one oracle run."""
    o = make(kind, sched)
    D, U, L, N, B, T, mv, E = 8, 32, 2, 100, 25, 4, -1.0, 18  # 72 steps
    X, Y = lstm_sequences(4, N, T, D, mv)
    rs = np.random.RandomState(5)
    perms = np.stack([rs.permutation(N) for _ in range(E)])
    w0 = kl.init_weights(D, U, L, seed=6)
    w64 = [a.astype(np.float64) for a in w0]
    with so.installed(o.learning_rate):
        h64, st = kl.fit(w64, "tanh", X, Y, E, B, perms, mv, adam=oo.state_for(w64, o, np.float64),
                         dtype=np.float64)
    net = _lstm(D, U, L, o, w0, mv)
    ha = net.fit(X, Y, epochs=7, batch_size=B, permutations=perms[:7], verbose=0).history["loss"]
    hb = net.fit(X, Y, epochs=E - 7, batch_size=B, permutations=perms[7:], verbose=0).history["loss"]
    hist = np.array(ha + hb)
    assert np.abs(hist - h64).max() <= 1e-4, (hist, h64)
    for a, b in zip(net.get_weights(), w64):
        assert np.abs(a - b).max() <= 2e-3
    assert net.get_optimizer_state()[2] == st.t == E * 4


# ---------------------------------------------------------------------------------------------- surfaces end to end
def test_batched_surface_with_device_labels():
    """A ragged batched fit labelled on the device (gamma=) under a schedule: per problem, the oracle fit of the
    problem alone with its own iterations."""
    from bore_b200 import BatchedMaximizableSequential, Dense, BinaryCrossentropy, sigmoid
    D, gamma = 6, 1 / 3
    ns, es = [150, 23, 64, 97], [8, 30, 0, 12]
    M = len(ns)
    dims, acts = [D, 32, 32, 1], ["elu", "elu", "linear"]
    rs = np.random.RandomState(10)
    X = [rs.uniform(size=(n, D)) for n in ns]
    y = [synthetic_targets(X[p]) + 0.3 * p * X[p][:, 0] for p in range(M)]
    o = layers.Adam(learning_rate=ExponentialDecay(1e-2, 12, 0.5))
    model = BatchedMaximizableSequential([Dense(32, activation="elu", input_dim=D), Dense(32, activation="elu"),
                                          Dense(1)], n_problems=M, transform=sigmoid, seed=1)
    model.compile(optimizer=o, loss=BinaryCrossentropy(from_logits=True))
    w0 = [km.init_weights(dims, 10 + p) for p in range(M)]
    model.set_weights(w0)
    draw = np.random.RandomState(1)  # the surface's permutations, as tests/test_gpu_ragged.py draws them
    for p in range(M):
        for fi, fo in zip(dims[:-1], dims[1:]):
            draw.uniform(size=(fi, fo))
    perms = [np.array([draw.permutation(ns[p]) for _ in range(es[p])], dtype=np.int64).reshape(es[p], ns[p])
             for p in range(M)]
    hist = model.fit(X, y, batch_size=64, epochs=es, gamma=gamma)
    got_w = model.get_weights()
    for p in range(M):
        z = y[p] < np.quantile(y[p], gamma)
        w = [a.copy() for a in w0[p]]
        with so.installed(o.learning_rate):
            h_ref, _ = km.fit(w, acts, X[p], z, es[p], 64, perms[p], adam=oo.state_for(w, o))
        assert np.abs(hist[p, :es[p]] - h_ref).max(initial=0) <= LOSS_TOL, p
        for a, b in zip(got_w[p], w):
            assert np.abs(a - b).max() <= 2e-3


def test_bore_end_to_end():
    import test_gpu_plugin as tgp
    from bore_b200.plugins.hpbandster import BORE

    def run():
        opt = BORE(tgp._space(), eta=3, min_budget=1 / 9, max_budget=1, seed=0, num_random_init=8,
                   num_steps_per_iter=200, num_starts=4, num_samples=256,
                   optimizer=layers.Adam(learning_rate=ExponentialDecay(1e-2, 50, 0.5)),
                   logger=logging.getLogger("bore-test"))
        return opt, opt.run(n_iterations=4, compute_fn=tgp._loss)

    opt, results = run()
    cg = opt.config_generator
    assert cg.logit is not None and cg.logit._last_stats["evals"] > 0
    assert isinstance(cg.logit._compiled["optimizer"].learning_rate, ExponentialDecay)
    _, again = run()
    assert [l for _, _, l in results] == [l for _, _, l in again]


def test_bore_hyperband_end_to_end():
    import test_gpu_lstm as tgl
    from bore_b200.plugins.hpbandster import BOREHyperband

    def run():
        opt = BOREHyperband(tgl._space(), eta=3, min_budget=1 / 9, max_budget=1, seed=0, num_random_init=6,
                            num_steps_per_iter=100, num_starts=4, num_samples=128,
                            optimizer=layers.Adam(learning_rate=ExponentialDecay(1e-2, 50, 0.5)),
                            logger=logging.getLogger("bore-mf-gpu"))
        return opt, opt.run(n_iterations=6, compute_fn=tgl._loss)

    opt, results = run()
    cg = opt.config_generator
    assert cg.funcs and all(f._last_stats["evals"] > 0 for f in cg.funcs.values())
    _, again = run()
    assert [l for _, _, l in results] == [l for _, _, l in again]
