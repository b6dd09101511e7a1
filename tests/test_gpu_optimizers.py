"""The optimizers RMSprop, Adagrad, Adadelta, Adamax and Nadam (and Adam with non-default hyper-parameters) on
the device, against the oracle (tests/optimizer_oracle.py) with the bars of tests/test_gpu_activations.py: every
fit kernel, both unit-split builds, many-model, weighted and ragged launches, an extended activation, the
optimizer state across calls and handles, the LSTM kernel and the plugins end to end."""
import logging

import numpy as np
import pytest

from oracle import keras_lstm as kl, keras_mlp as km
import optimizer_oracle as oo
import weighted_oracle as wo
from helpers import lstm_factory, lstm_sequences, synthetic_targets
from bore_b200 import layers

pytestmark = pytest.mark.gpu

LOSS_TOL = 1e-4

CONFIGS = {
    "rmsprop": dict(),
    "rmsprop_centered": dict(centered=True),
    "rmsprop_momentum": dict(momentum=0.9),
    "rmsprop_custom": dict(learning_rate=5e-3, rho=0.8, epsilon=1e-5),
    "adagrad": dict(),
    "adagrad_custom": dict(learning_rate=2e-2, initial_accumulator_value=0.5),
    "adadelta": dict(),
    "adadelta_custom": dict(learning_rate=1.0, rho=0.9, epsilon=1e-6),
    "adamax": dict(),
    "adamax_custom": dict(learning_rate=3e-3, beta_1=0.8, beta_2=0.99),
    "nadam": dict(),
    "nadam_custom": dict(learning_rate=3e-3, beta_1=0.85, beta_2=0.99),
}


@pytest.fixture(autouse=True, scope="module")
def _optimizer_oracle():
    with oo.installed():
        yield


def make(name):
    return type(layers.optimizer_spec(name.split("_")[0]))(**CONFIGS[name])


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
    h, st = km.fit(w, acts, X, z, E, 64, perms, adam=st, l2=l2)
    return h, w, st


DIMS, ACTS = [6, 32, 32, 1], ["elu", "elu", "sigmoid"]


@pytest.mark.parametrize("mode", [1, 2, 3, 4])
@pytest.mark.parametrize("name", sorted(CONFIGS))
@pytest.mark.parametrize("l2", [0.0, 1e-3])
def test_fit_modes(name, mode, l2):
    o = make(name)
    N, E = 333, 12
    X, z, perms = _problem(DIMS, N, E, seed=5)
    w0 = km.init_weights(DIMS, 3)
    h_ref, w_ref, st = _oracle_fit(w0, ACTS, X, z, E, perms, o, l2)
    net = _net(DIMS, ACTS, o, w0)
    net.set_fit_mode(mode)
    hist = net.fit(X, z, E, 64, perms, l2=l2)
    assert np.abs(hist - h_ref).max() <= LOSS_TOL, np.abs(hist - h_ref).max()
    for a, b in zip(net.get_weights(), w_ref):
        assert np.abs(a - b).max() <= 2e-3
    state = net.get_optimizer_state()
    assert state[2] == st.t == E * 6
    if o.kind == "nadam":
        assert abs(state[3] - st.cache) <= 1e-6 * abs(st.cache)


@pytest.mark.parametrize("dims", [[50, 64, 64, 64, 1], [6, 32, 32, 1], [6, 16, 16, 1], [7, 24, 24, 1],
                                  [7, 40, 40, 1]])
@pytest.mark.parametrize("name", ["nadam", "rmsprop_momentum", "adagrad_custom"])
def test_unit_split_builds(dims, name):
    """Fit mode 4: hidden widths 16 / 32 / 64 take the compile-time builds of the unit-split kernel, 24 / 40 its
    run-time build."""
    o = make(name)
    acts = ["tanh"] * (len(dims) - 2) + ["sigmoid"]
    N, E = 700, 4
    X, z, perms = _problem(dims, N, E, seed=9)
    w0 = km.init_weights(dims, 4)
    h_ref, w_ref, _ = _oracle_fit(w0, acts, X, z, E, perms, o)
    net = _net(dims, acts, o, w0)
    net.set_fit_mode(4)
    assert np.abs(net.fit(X, z, E, 64, perms) - h_ref).max() <= LOSS_TOL
    for a, b in zip(net.get_weights(), w_ref):
        assert np.abs(a - b).max() <= 2e-3


@pytest.mark.parametrize("M", [20, 600])
@pytest.mark.parametrize("name", ["adamax", "nadam", "adadelta_custom"])
def test_many_models(M, name):
    o = make(name)
    N, E = 150, 6
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


@pytest.mark.parametrize("name", ["rmsprop_centered", "nadam"])
def test_weighted_fit(name):
    o = make(name)
    N, E = 200, 10
    X, z, perms = _problem(DIMS, N, E, seed=11)
    sw = np.random.RandomState(12).uniform(0, 2, size=N).astype(np.float32)
    w0 = km.init_weights(DIMS, 6)
    w_ref = [a.copy() for a in w0]
    h_ref, _ = wo.fit(w_ref, ACTS, X, z, E, 64, perms, sample_weight=sw, class_weight={0: 0.5, 1: 2.0},
                      adam=oo.state_for(w_ref, o))
    for mode in (1, 2, 4):
        net = _net(DIMS, ACTS, o, w0)
        net.set_fit_mode(mode)
        hist = net.fit(X, z, E, 64, perms, w=sw, class_weight=(0.5, 2.0))
        assert np.abs(hist - h_ref).max() <= LOSS_TOL, mode


@pytest.mark.parametrize("name", ["adagrad", "adamax_custom"])
def test_ragged_fit(name):
    from bore_b200.ragged import RaggedLayout
    o = make(name)
    n, e = np.array([40, 130, 75]), np.array([9, 3, 5])
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
        h_ref, _, _ = _oracle_fit(ws[p], ACTS, probs[p][0], probs[p][1], int(e[p]), probs[p][2], o)
        assert np.abs(loss[lay.losses[p]:lay.losses[p + 1]] - h_ref).max() <= LOSS_TOL, p


@pytest.mark.parametrize("mode", [1, 2, 3, 4])
def test_extended_activation(mode):
    import activation_oracle as ao
    o = make("nadam")
    dims, acts = [6, 32, 32, 1], ["softplus", "selu", "sigmoid"]
    N, E = 200, 8
    X, z, perms = _problem(dims, N, E, seed=13)
    w0 = km.init_weights(dims, 7)
    with ao.installed():
        h_ref, _, _ = _oracle_fit(w0, acts, X, z, E, perms, o)
    net = _net(dims, acts, o, w0)
    net.set_fit_mode(mode)
    assert np.abs(net.fit(X, z, E, 64, perms) - h_ref).max() <= LOSS_TOL


@pytest.mark.parametrize("name", ["nadam", "adagrad", "rmsprop_momentum"])
def test_two_fits_follow_one_oracle_run(name):
    o = make(name)
    N, E = 200, 10
    X, z, perms = _problem(DIMS, N, E, seed=14)
    w0 = km.init_weights(DIMS, 8)
    h_ref, w_ref, st = _oracle_fit(w0, ACTS, X, z, E, perms, o)
    net = _net(DIMS, ACTS, o, w0)
    ha = net.fit(X, z, 4, 64, perms[:4])
    hb = net.fit(X, z, E - 4, 64, perms[4:])
    assert np.abs(np.concatenate([ha, hb]) - h_ref).max() <= LOSS_TOL
    for a, b in zip(net.get_weights(), w_ref):
        assert np.abs(a - b).max() <= 2e-3


@pytest.mark.parametrize("name", ["nadam", "adagrad_custom", "adadelta"])
def test_state_round_trip_is_bit_identical(name):
    """get -> set onto a fresh handle: the next fit continues exactly like the uninterrupted handle."""
    o = make(name)
    N, E = 200, 6
    X, z, perms = _problem(DIMS, N, E, seed=15)
    w0 = km.init_weights(DIMS, 9)
    a = _net(DIMS, ACTS, o, w0)
    a.fit(X, z, 3, 64, perms[:3])
    state = a.get_optimizer_state()
    assert len(state) == (4 if o.kind == "nadam" else 3)
    b = _net(DIMS, ACTS, o, [np.array(w) for w in a.get_weights()])
    b.set_optimizer_state(*state)
    ha, hb = a.fit(X, z, 3, 64, perms[3:]), b.fit(X, z, 3, 64, perms[3:])
    assert np.array_equal(ha, hb)
    for u, v in zip(a.get_weights(), b.get_weights()):
        assert np.array_equal(u, v)
    for u, v in zip(a.get_optimizer_state(), b.get_optimizer_state()):
        assert all(np.array_equal(p, q) for p, q in zip(u, v)) if isinstance(u, list) else u == v


def test_reset_and_kind_change():
    N, E = 100, 2
    X, z, perms = _problem(DIMS, N, E, seed=16)
    net = _net(DIMS, ACTS, make("adagrad_custom"), km.init_weights(DIMS, 10), n_models=2)
    s0, s1, it = net.get_optimizer_state(model=1)
    assert it == 0 and all(np.all(a == np.float32(0.5)) for a in s0) and all(np.all(a == 0) for a in s1)
    net.fit(X, z, E, 64, perms, model=1)
    assert net.get_optimizer_state(model=1)[2] == 4
    net.reset_optimizer()
    s0, s1, it = net.get_optimizer_state(model=1)
    assert it == 0 and all(np.all(a == np.float32(0.5)) for a in s0) and all(np.all(a == 0) for a in s1)
    net.fit(X, z, E, 64, perms, model=0)
    net.set_optimizer_kind(make("nadam"))  # a new kind: every model starts over
    for m in range(2):
        s0, s1, it, cache = net.get_optimizer_state(model=m)
        assert it == 0 and cache == 1.0 and all(np.all(a == 0) for a in s0 + s1)
    net.fit(X, z, E, 64, perms, model=0)
    assert net.get_optimizer_state(model=0)[3] < 1.0
    net.reset_optimizer(0, 1)
    assert net.get_optimizer_state(model=0)[3] == 1.0
    net.set_optimizer_kind(make("nadam_custom"))  # same kind: hyper-parameters only, the state stays
    net.fit(X, z, E, 64, perms, model=0)
    assert net.get_optimizer_state(model=0)[2] == 4


@pytest.mark.parametrize("name", sorted(CONFIGS) + ["adam_custom"])
def test_lstm(name):
    """The LSTM fit kernel under every kind against keras_lstm with the optimizer oracle, with the bars of
    tests/test_gpu_lstm.py; two fit calls, the state persists between them."""
    from bore_b200.layers import BinaryCrossentropy
    o = make(name) if name != "adam_custom" else layers.Adam(learning_rate=3e-3, beta_1=0.8, beta_2=0.99,
                                                             epsilon=1e-6)
    D, U, L, N, B, T, mv, E = 8, 32, 2, 100, 64, 4, -1.0, 12
    X, Y = lstm_sequences(4, N, T, D, mv)
    rs = np.random.RandomState(5)
    perms = np.stack([rs.permutation(N) for _ in range(E)])
    w0 = kl.init_weights(D, U, L, seed=6)
    w64 = [a.astype(np.float64) for a in w0]
    h64, st = kl.fit(w64, "tanh", X, Y, E, B, perms, mv, adam=oo.state_for(w64, o, np.float64), dtype=np.float64)
    net = lstm_factory(D, U, L, "tanh").build_many_to_many(mask_value=mv)
    net.compile(optimizer=o, loss=BinaryCrossentropy(from_logits=True))
    net.set_weights(w0)
    ha = net.fit(X, Y, epochs=6, batch_size=B, permutations=perms[:6], verbose=0).history["loss"]
    hb = net.fit(X, Y, epochs=E - 6, batch_size=B, permutations=perms[6:], verbose=0).history["loss"]
    hist = np.array(ha + hb)
    assert np.abs(hist - h64).max() <= 1e-4, (hist, h64)
    for a, b in zip(net.get_weights(), w64):
        assert np.abs(a - b).max() <= 2e-3
    state = net.get_optimizer_state()
    assert state[2] == st.t == E * 2
    if o.kind == "nadam":
        assert abs(state[3] - st.cache) <= 1e-6


def _bore_run(optimizer, seed):
    import test_gpu_plugin as tgp
    from bore_b200.plugins.hpbandster import BORE
    opt = BORE(tgp._space(), eta=3, min_budget=1 / 9, max_budget=1, seed=seed, num_random_init=8,
               num_steps_per_iter=200, num_starts=4, num_samples=256, optimizer=optimizer,
               logger=logging.getLogger("bore-test"))
    return opt, opt.run(n_iterations=4, compute_fn=tgp._loss)


def _in_bounds(results, space):
    for cfg, _, _ in results:
        for hp in space.get_hyperparameters():
            if hasattr(hp, "lower"):
                assert hp.lower <= cfg[hp.name] <= hp.upper


def test_bore_rmsprop_end_to_end():
    import test_gpu_plugin as tgp
    opt, results = _bore_run("rmsprop", 0)
    cg = opt.config_generator
    assert cg.logit is not None and cg.logit._last_stats["evals"] > 0
    assert cg.logit._compiled["optimizer"].kind == "rmsprop"
    _in_bounds(results, tgp._space())
    _, again = _bore_run("rmsprop", 0)
    assert [l for _, _, l in results] == [l for _, _, l in again]


def test_bore_hyperband_nadam_end_to_end():
    import test_gpu_lstm as tgl
    from bore_b200.plugins.hpbandster import BOREHyperband

    def run():
        opt = BOREHyperband(tgl._space(), eta=3, min_budget=1 / 9, max_budget=1, seed=0, num_random_init=6,
                            num_steps_per_iter=100, num_starts=4, num_samples=128, optimizer="nadam",
                            logger=logging.getLogger("bore-mf-gpu"))
        return opt, opt.run(n_iterations=6, compute_fn=tgl._loss)

    opt, results = run()
    cg = opt.config_generator
    assert cg.funcs and all(f._last_stats["evals"] > 0 for f in cg.funcs.values())
    _in_bounds(results, tgl._space())
    _, again = run()
    assert [l for _, _, l in results] == [l for _, _, l in again]


def test_batched_adagrad():
    from bore_b200 import BatchedMaximizableSequential, Dense

    def run():
        M, D = 6, 4
        model = BatchedMaximizableSequential([Dense(16, activation="relu", input_dim=D), Dense(16, activation="relu"),
                                              Dense(1, activation="sigmoid")], n_problems=M, seed=2)
        model.compile(optimizer="adagrad", loss="binary_crossentropy")
        rs = np.random.RandomState(1)
        X = rs.uniform(size=(M, 80, D))
        y = np.sum((X - 0.4) ** 2, axis=2)
        z = (y < np.quantile(y, 0.3, axis=1, keepdims=True)).astype(np.float32)
        hist = model.fit(X, z, batch_size=32, epochs=5)
        assert np.all(np.isfinite(hist))
        return model.argmax([(0.0, 1.0)] * D, num_starts=4, num_samples=128, random_state=0)

    a, b = run(), run()
    for p in range(len(a)):
        assert a[p] is not None and np.all(a[p].x >= 0) and np.all(a[p].x <= 1)
        assert np.array_equal(a[p].x, b[p].x)
