"""Keras Dropout between Dense layers on the device, against the oracle (tests/dropout_oracle.py) with the bars of
tests/test_gpu_regularizers.py (loss trajectory 1e-4, weights 2e-3): every fit mode, both unit-split builds, many-model,
weighted and ragged launches, another optimizer with a schedule and l1, continued fits, the masks bit for bit through
the public path, hard_sigmoid's act' at saturation, Dropout(0.0) bit-identical to none, and the Sequential and batched surfaces, whose inference is
bit-identical to the same weights without Dropout layers."""
import numpy as np
import pytest
from scipy.optimize import Bounds

from oracle import keras_mlp as km
import dropout_oracle as do
import optimizer_oracle as oo
import regularizer_oracle as ro
import schedule_oracle as so
from helpers import synthetic_targets
from bore_b200 import layers, schedules
from bore_b200.layers import Dense, Dropout

pytestmark = pytest.mark.gpu

LOSS_TOL = 1e-4
W_TOL = 2e-3
DIMS = [6, 32, 32, 1]


@pytest.fixture(autouse=True, scope="module")
def _oracles():
    with oo.installed():
        yield


def _problem(dims, N, E, seed):
    rs = np.random.RandomState(seed)
    X = rs.uniform(size=(N, dims[0]))
    y = synthetic_targets(X)
    return X, (y < np.quantile(y, 0.25)).astype(np.float32), np.stack([rs.permutation(N) for _ in range(E)])


def _net(dims, acts, w=None, n_models=1, opt=None, rates=None, seeds=None):
    from bore_b200.engine import NativeMLP
    net = NativeMLP(dims, acts, n_models=n_models)
    if opt is not None:
        net.set_optimizer_kind(opt)
    if w is not None:
        for i in range(n_models):
            net.set_weights(w, model=i)
    if rates is not None:
        net.set_dropout(rates, seeds)
    return net


def _oracle_fit(w0, acts, X, z, E, perms, rates, seeds, model=0, opt=None, l2=0.0, sw=None, state=None, B=64):
    w = [a.copy() for a in w0]
    st = state if state is not None else km.AdamState(w) if opt is None else oo.state_for(w, opt)
    h, st = do.fit(w, acts, X, z, E, B, perms, rates, seeds, model=model, state=st, l2=l2, sample_weight=sw)
    return h, w, st


def _close(hist, h_ref, ws, w_ref):
    assert np.abs(hist - h_ref).max() <= LOSS_TOL, np.abs(hist - h_ref).max()
    for a, b in zip(ws, w_ref):
        assert np.abs(a - b).max() <= W_TOL, np.abs(a - b).max()


@pytest.mark.parametrize("mode", [1, 2, 3, 4])
@pytest.mark.parametrize("rate", [0.1, 0.5])
@pytest.mark.parametrize("act", ["relu", "elu", "selu"])
def test_fit_modes(act, rate, mode):
    import activation_oracle as ao
    acts = [act, act, "sigmoid"]
    N, E = 333, 10
    X, z, perms = _problem(DIMS, N, E, seed=5)
    w0 = km.init_weights(DIMS, 3)
    rates, seeds = [rate, rate], [17, 2 ** 31 + 5]
    with ao.installed():
        h_ref, w_ref, _ = _oracle_fit(w0, acts, X, z, E, perms, rates, seeds)
    net = _net(DIMS, acts, w0, rates=rates, seeds=seeds)
    net.set_fit_mode(mode)
    _close(net.fit(X, z, E, 64, perms), h_ref, net.get_weights(), w_ref)


@pytest.mark.parametrize("dims", [[50, 64, 64, 64, 1], [6, 32, 32, 1], [6, 16, 16, 1], [7, 24, 24, 1],
                                  [7, 40, 40, 1]])
def test_unit_split_builds(dims):
    """Fit mode 4: hidden widths 16 / 32 / 64 take the compile-time builds of the unit-split kernel, 24 / 40 its
    run-time build."""
    acts = ["tanh"] * (len(dims) - 2) + ["sigmoid"]
    N, E = 700, 4
    X, z, perms = _problem(dims, N, E, seed=9)
    w0 = km.init_weights(dims, 4)
    rates = [0.2 + 0.1 * i for i in range(len(dims) - 2)]
    seeds = [100 + i for i in range(len(rates))]
    h_ref, w_ref, _ = _oracle_fit(w0, acts, X, z, E, perms, rates, seeds)
    net = _net(dims, acts, w0, rates=rates, seeds=seeds)
    net.set_fit_mode(4)
    _close(net.fit(X, z, E, 64, perms), h_ref, net.get_weights(), w_ref)


@pytest.mark.parametrize("M", [20, 600])
def test_many_models(M):
    """Every model of a launch has its own masks (its model index); two models with the same data and weights end
    with different weights."""
    acts = ["elu", "elu", "sigmoid"]
    N, E = 150, 6
    probs = [_problem(DIMS, N, E, seed=50 + i) for i in range(M)]
    probs[1] = probs[0]
    ws = [km.init_weights(DIMS, 200 + i) for i in range(M)]
    ws[1] = ws[0]
    rates, seeds = [0.3, 0.2], [5, 6]
    net = _net(DIMS, acts, n_models=M, rates=rates, seeds=seeds)
    for i, w in enumerate(ws):
        net.set_weights(w, model=i)
    Xd = net.to_device(np.concatenate([p[0] for p in probs]), np.float32)
    zd = net.to_device(np.concatenate([p[1] for p in probs]).astype(np.float32), np.float32)
    pd = net.to_device(np.stack([p[2] for p in probs]).astype(np.int32), np.int32)
    loss = net.fit_dev(Xd, zd, N, 64, E, pd, model0=0, count=M, shared_data=False, shared_perm=False).cpu().numpy()
    for i in sorted(set(list(range(0, M, max(1, M // 25))) + [1, M - 1])):
        h_ref, w_ref, _ = _oracle_fit(ws[i], acts, probs[i][0], probs[i][1], E, probs[i][2], rates, seeds, model=i)
        _close(loss[i], h_ref, net.get_weights(model=i), w_ref)
    assert not np.array_equal(net.get_weights(model=0)[0], net.get_weights(model=1)[0])


def test_weighted_fit():
    acts = ["relu", "relu", "sigmoid"]
    N, E = 200, 10
    X, z, perms = _problem(DIMS, N, E, seed=11)
    sw = np.random.RandomState(12).uniform(0, 2, size=N).astype(np.float32)
    w0 = km.init_weights(DIMS, 6)
    rates, seeds = [0.25, 0.4], [1, 2]
    h_ref, w_ref, _ = _oracle_fit(w0, acts, X, z, E, perms, rates, seeds, sw=sw)
    for mode in (1, 2, 3, 4):
        net = _net(DIMS, acts, w0, rates=rates, seeds=seeds)
        net.set_fit_mode(mode)
        _close(net.fit(X, z, E, 64, perms, w=sw), h_ref, net.get_weights(), w_ref)


def test_ragged_fit():
    from bore_b200.ragged import RaggedLayout
    acts = ["elu", "elu", "sigmoid"]
    n, e = np.array([40, 130, 75]), np.array([9, 3, 5])
    lay = RaggedLayout(n, e)
    probs = [_problem(DIMS, int(n[p]), int(e[p]), seed=20 + p) for p in range(3)]
    ws = [km.init_weights(DIMS, 30 + p) for p in range(3)]
    rates, seeds = [0.5, 0.1], [7, 8]
    net = _net(DIMS, acts, n_models=3, rates=rates, seeds=seeds)
    for p, w in enumerate(ws):
        net.set_weights(w, model=p)
    Xd = net.to_device(np.concatenate([p[0] for p in probs]), np.float32)
    zd = net.to_device(np.concatenate([p[1] for p in probs]).astype(np.float32), np.float32)
    pd = net.to_device(np.concatenate([p[2].reshape(-1) for p in probs]).astype(np.int32), np.int32)
    loss = net.fit_ragged_dev(Xd, zd, lay, 64, pd).cpu().numpy()
    for p in range(3):
        h_ref, w_ref, _ = _oracle_fit(ws[p], acts, probs[p][0], probs[p][1], int(e[p]), probs[p][2], rates, seeds,
                                      model=p)
        _close(loss[lay.losses[p]:lay.losses[p + 1]], h_ref, net.get_weights(model=p), w_ref)


@pytest.mark.parametrize("mode", [1, 2, 3, 4])
def test_rmsprop_schedule_l1(mode):
    acts = ["elu", "elu", "sigmoid"]
    sched = schedules.ExponentialDecay(1e-3, decay_steps=5, decay_rate=0.8)
    opt = layers.RMSprop(learning_rate=sched)
    N, E = 200, 8
    X, z, perms = _problem(DIMS, N, E, seed=14)
    w0 = km.init_weights(DIMS, 8)
    l1 = [1e-3] * len(w0)
    rates, seeds = [0.3, 0.3], [11, 12]
    with so.installed(sched):
        h_ref, w_ref, _ = _oracle_fit(w0, acts, X, z, E, perms, rates, seeds, opt=opt, l2=ro.Factors(0.0, l1))
    net = _net(DIMS, acts, w0, opt=opt, rates=rates, seeds=seeds)
    net.set_fit_mode(mode)
    _close(net.fit(X, z, E, 64, perms, l2=[0.0] * len(w0), l1=l1), h_ref, net.get_weights(), w_ref)


@pytest.mark.parametrize("mode", [1, 2, 3, 4])
def test_continued_fits(mode):
    """A second fit continues the mask stream; a fit from set_optimizer_state(iterations=k) reproduces it."""
    acts = ["relu", "relu", "sigmoid"]
    N, E = 200, 4
    X, z, perms = _problem(DIMS, N, 2 * E, seed=15)
    w0 = km.init_weights(DIMS, 9)
    rates, seeds = [0.4, 0.2], [3, 4]
    h1, w1, st = _oracle_fit(w0, acts, X, z, E, perms[:E], rates, seeds)
    h2, w2, st = _oracle_fit(w1, acts, X, z, E, perms[E:], rates, seeds, state=st)
    net = _net(DIMS, acts, w0, rates=rates, seeds=seeds)
    net.set_fit_mode(mode)
    _close(net.fit(X, z, E, 64, perms[:E]), h1, net.get_weights(), w1)
    _close(net.fit(X, z, E, 64, perms[E:]), h2, net.get_weights(), w2)
    # the same second fit from the oracle's state after the first
    net2 = _net(DIMS, acts, w1, rates=rates, seeds=seeds)
    net2.set_fit_mode(mode)
    st1 = _oracle_fit(w0, acts, X, z, E, perms[:E], rates, seeds)[2]
    net2.set_optimizer_state(st1.m, st1.v, st1.t)
    _close(net2.fit(X, z, E, 64, perms[E:]), h2, net2.get_weights(), w2)


@pytest.mark.parametrize("mode", [1, 2, 3, 4])
def test_masks_bit_exact(mode):
    """One step from zero slots at iterations t with sample weights one-hot at minibatch position i: a parameter is
    left bit-unchanged exactly where the oracle's gradient (same masks) is exactly zero (relu: act' is exact)."""
    dims, acts = [5, 20, 12, 1], ["relu", "relu", "sigmoid"]
    B = 40
    M = 3
    X, z, _ = _problem(dims, B, 1, seed=16)
    rates, seeds = [0.5, 0.3], [2024, 99]
    perm = np.random.RandomState(17).permutation(B)[None]
    w0s = [km.init_weights(dims, 40 + m) for m in range(M)]
    zero = [np.zeros_like(a) for a in w0s[0]]
    for t, i in ((0, 0), (1, 7), (12345, 39), (2 ** 32 + 3, 21)):
        onehot = np.zeros(B, np.float32)
        onehot[perm[0, i]] = 1.0
        net = _net(dims, acts, n_models=M, rates=rates, seeds=seeds)
        net.set_fit_mode(mode)
        for m in range(M):
            net.set_weights(w0s[m], model=m)
            net.set_optimizer_state(zero, zero, t, model=m)
        # model 0 alone, then a batched launch of models 1 and 2 (model index > 0 inside one launch)
        net.fit(X, z, 1, B, perm, model=0, w=onehot)
        Xd, zd = net.to_device(X, np.float32), net.to_device(z, np.float32)
        wd = net.to_device(onehot, np.float32)
        net.fit_dev(Xd, zd, B, B, 1, net.to_device(perm.astype(np.int32), np.int32), model0=1, count=2, w_dev=wd)
        for m in range(M):
            idx = perm[0]
            masks = [do.keep_mask(l, t, B, dims[l + 1], r, s, m) for l, (r, s) in enumerate(zip(rates, seeds))]
            _, g = do.loss_and_weight_grads(w0s[m], acts, X[idx].astype(np.float32), z[idx], masks, rates,
                                            sample_weight=onehot[idx])
            got = net.get_weights(model=m)
            for a, b, gg in zip(got, w0s[m], g):
                unchanged = np.asarray(a) == b
                assert np.array_equal(unchanged, gg == 0), (t, i, m)
            assert any((gg == 0).any() for gg in g[:4]) and all((gg != 0).any() for gg in g)


def _saturating_weights(dims, seed):
    """Glorot hidden-layer weights times 12: about half the hard_sigmoid pre-activations lie beyond +-2.5, where h is
    exactly 0 or 1.  The output layer keeps its scale, so the logit does not saturate and no gradient is so small that
    Adam's first step (about lr per parameter) would vanish in the rounding of the weight."""
    ws = km.init_weights(dims, seed)
    return [a * np.float32(12.0) if i < len(ws) - 2 else a for i, a in enumerate(ws)]


@pytest.mark.parametrize("mode", [1, 2, 3, 4])
@pytest.mark.parametrize("rate", [0.11, 0.46])
def test_hard_sigmoid_saturated(rate, mode):
    """hard_sigmoid's act' is 0 at h = 1.  At these rates fl32(fp32(scale) fp32(1 - rate)) is 1 - ulp, so recovering h
    from h~ by that product would give act' = 0.2 on every kept saturated unit.  Two checks: one step from zero slots
    with one-hot sample weights, where a parameter must stay bit-unchanged exactly where the oracle's gradient is
    exactly 0 (act' of hard_sigmoid is exact); and a whole fit against the oracle."""
    import activation_oracle as ao
    dims, acts = [5, 20, 12, 1], ["hard_sigmoid", "hard_sigmoid", "sigmoid"]
    assert np.float32(np.float32(1.0 / (1.0 - float(np.float32(rate)))) * np.float32(1.0 - np.float32(rate))) < 1
    B = 40
    X, z, _ = _problem(dims, B, 1, seed=30)
    rates, seeds = [rate, rate], [5, 6]
    perm = np.random.RandomState(31).permutation(B)[None]
    w0 = _saturating_weights(dims, 32)
    zero = [np.zeros_like(a) for a in w0]
    with ao.installed():
        h1 = km.forward(w0, acts, X[perm[0]], keep=True)[1][1]
        for i in (3, 17, 38):
            onehot = np.zeros(B, np.float32)
            onehot[perm[0, i]] = 1.0
            net = _net(dims, acts, w0, rates=rates, seeds=seeds)
            net.set_fit_mode(mode)
            net.set_optimizer_state(zero, zero, 9)
            net.fit(X, z, 1, B, perm, w=onehot)
            masks = [do.keep_mask(l, 9, B, dims[l + 1], r, s, 0) for l, (r, s) in enumerate(zip(rates, seeds))]
            _, g = do.loss_and_weight_grads(w0, acts, X[perm[0]].astype(np.float32), z[perm[0]], masks, rates,
                                            sample_weight=onehot[perm[0]])
            assert np.sum((h1[i] == 1.0) & (masks[0][i] == 1)) >= 2  # kept saturated units of this sample
            for a, b, gg in zip(net.get_weights(), w0, g):
                assert np.array_equal(np.asarray(a) == b, gg == 0), i
        N, E = 200, 6
        X, z, perms = _problem(dims, N, E, seed=33)
        h_ref, w_ref, _ = _oracle_fit(w0, acts, X, z, E, perms, rates, seeds)
    net = _net(dims, acts, w0, rates=rates, seeds=seeds)
    net.set_fit_mode(mode)
    _close(net.fit(X, z, E, 64, perms), h_ref, net.get_weights(), w_ref)


@pytest.mark.parametrize("mode", [1, 2, 3, 4])
def test_rate_zero_bit_identical(mode):
    acts = ["elu", "elu", "sigmoid"]
    N, E = 200, 4
    X, z, perms = _problem(DIMS, N, E, seed=18)
    w0 = km.init_weights(DIMS, 10)
    a = _net(DIMS, acts, w0)
    b = _net(DIMS, acts, w0, rates=[0.0, 0.0], seeds=[1, 2])
    for net in (a, b):
        net.set_fit_mode(mode)
    ha, hb = a.fit(X, z, E, 64, perms), b.fit(X, z, E, 64, perms)
    assert np.array_equal(ha, hb)
    assert all(np.array_equal(x, y) for x, y in zip(a.get_weights(), b.get_weights()))

    from bore_b200.models import Sequential
    outs = []
    for drop in (False, True):
        m = Sequential(seed=3)
        m.add(Dense(32, activation="elu", input_dim=6))
        if drop:
            m.add(Dropout(0.0))
        m.add(Dense(32, activation="elu"))
        m.add(Dense(1, activation="sigmoid"))
        m.compile(optimizer="adam", loss="binary_crossentropy")
        m._engine(6).set_fit_mode(mode)
        h = m.fit(X, z, batch_size=64, epochs=E, verbose=0).history["loss"]
        outs.append((h, m.get_weights()))
    assert outs[0][0] == outs[1][0] and all(np.array_equal(x, y) for x, y in zip(outs[0][1], outs[1][1]))


def _sequential(drop, seed=1):
    from bore_b200.models import MaximizableSequential
    m = MaximizableSequential(seed=seed)
    m.add(Dense(32, activation="elu", input_dim=6))
    if drop:
        m.add(Dropout(0.3, seed=77))
    m.add(Dense(32, activation="elu"))
    if drop:
        m.add(Dropout(0.2, seed=78))
    m.add(Dense(1, activation="sigmoid"))
    m.compile(optimizer="adam", loss="binary_crossentropy", metrics=["accuracy"])
    return m


@pytest.mark.parametrize("mode", [1, 4])
def test_sequential_surface(mode):
    """fit applies the Dropout; predict, evaluate, value_and_gradient and argmax are those of the same weights
    without Dropout layers, bit for bit."""
    acts = ["elu", "elu", "sigmoid"]
    N, E = 200, 6
    X, z, perms = _problem(DIMS, N, E, seed=19)
    w0 = km.init_weights(DIMS, 11)
    m = _sequential(True)
    m.set_weights(w0)
    m._engine(6).set_fit_mode(mode)
    hist = np.array(m.fit(X, z, batch_size=64, epochs=E, permutations=perms, verbose=0).history["loss"])
    h_ref, w_ref, _ = _oracle_fit(w0, acts, X, z, E, perms, [0.3, 0.2], [77, 78])
    _close(hist, h_ref, m.get_weights(), w_ref)
    plain = _sequential(False)
    plain.set_weights(m.get_weights())
    Xq = np.random.RandomState(20).uniform(size=(300, 6))
    assert np.array_equal(m.predict(Xq), plain.predict(Xq))
    assert m.evaluate(X, z) == plain.evaluate(X, z)
    for ga, gb in zip(m._native_value_and_grad(Xq, "sigmoid", True), plain._native_value_and_grad(Xq, "sigmoid", True)):
        assert np.array_equal(np.asarray(ga), np.asarray(gb))
    b = Bounds(np.zeros(6), np.ones(6))
    ra = m.argmax(b, num_starts=4, num_samples=256, print_fn=None, random_state=np.random.RandomState(5))
    rb = plain.argmax(b, num_starts=4, num_samples=256, print_fn=None, random_state=np.random.RandomState(5))
    assert np.array_equal(ra.x, rb.x) and ra.fun == rb.fun


def test_batched_surface():
    from bore_b200 import BatchedMaximizableSequential, BinaryCrossentropy, sigmoid
    M, N, D, E = 4, 150, 6, 6
    dims, acts = [D, 32, 32, 1], ["elu", "elu", "linear"]
    rs = np.random.RandomState(21)
    X = rs.uniform(size=(M, N, D))
    z = np.stack([(synthetic_targets(x) < np.quantile(synthetic_targets(x), 0.3)).astype(np.float32) for x in X])
    perms = np.stack([rs.permutation(N) for _ in range(E)])

    def make(drop):
        ls = [Dense(32, activation="elu", input_dim=D)] + ([Dropout(0.25, seed=5)] if drop else []) + \
             [Dense(32, activation="elu")] + ([Dropout(0.5, seed=6)] if drop else []) + [Dense(1)]
        model = BatchedMaximizableSequential(ls, n_problems=M, transform=sigmoid, seed=1)
        model.compile(optimizer="adam", loss=BinaryCrossentropy(from_logits=True))
        return model

    w0 = [km.init_weights(dims, 10 + p) for p in range(M)]
    model = make(True)
    model.set_weights(w0)
    hist = model.fit(X, z, batch_size=64, epochs=E, permutations=perms)
    got = model.get_weights()
    for p in range(M):
        h_ref, w_ref, _ = _oracle_fit(w0[p], acts, X[p], z[p], E, perms, [0.25, 0.5], [5, 6], model=p)
        _close(np.asarray(hist[p]), h_ref, got[p], w_ref)
    plain = make(False)
    plain.set_weights(got)
    Xq = rs.uniform(size=(M, 100, D))
    assert np.array_equal(model.predict(Xq), plain.predict(Xq))
    b = Bounds(np.zeros(D), np.ones(D))
    ra = model.argmax(b, num_starts=4, num_samples=256, random_state=np.random.RandomState(5))
    rb = plain.argmax(b, num_starts=4, num_samples=256, random_state=np.random.RandomState(5))
    for p in range(M):
        assert (ra[p] is None) == (rb[p] is None)
        if ra[p] is not None:
            assert np.array_equal(ra[p].x, rb[p].x) and ra[p].fun == rb[p].fun
