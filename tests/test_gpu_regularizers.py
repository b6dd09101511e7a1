"""Keras l1 and l1_l2 regularisation on the device, against the oracle (tests/regularizer_oracle.py) with the bars of
tests/test_gpu_optimizers.py (loss trajectory 1e-4, weights 2e-3): every fit kernel, both unit-split builds, many-model,
weighted and ragged launches, an extended activation, other optimizers, evaluate, the LSTM, the batched surface, the
bit-exact l1 = 0 path and the native argument checks."""
import ctypes as C

import numpy as np
import pytest

from oracle import keras_lstm as kl, keras_mlp as km
import optimizer_oracle as oo
import regularizer_oracle as ro
import weighted_oracle as wo
from helpers import lstm_factory, lstm_sequences, synthetic_targets
from bore_b200 import layers

pytestmark = pytest.mark.gpu

LOSS_TOL = 1e-4
W_TOL = 2e-3
DIMS, ACTS = [6, 32, 32, 1], ["elu", "elu", "sigmoid"]


@pytest.fixture(autouse=True, scope="module")
def _oracles():
    with oo.installed(), ro.installed():
        yield


def _factors(case, n):
    """Per-array (l2, l1) factors in Keras order [k0, b0, k1, b1, ...]."""
    if case == "l1":
        return [0.0] * n, [1e-3] * n
    if case == "l1_l2":
        return [1e-3] * n, [2e-3] * n
    assert case == "bias_l1"
    return [0.0] * n, [0.0 if i % 2 == 0 else 5e-3 for i in range(n)]


def _problem(dims, N, E, seed):
    rs = np.random.RandomState(seed)
    X = rs.uniform(size=(N, dims[0]))
    y = synthetic_targets(X)
    return X, y < np.quantile(y, 0.25), np.stack([rs.permutation(N) for _ in range(E)])


def _net(dims, acts, w=None, n_models=1, opt=None):
    from bore_b200.engine import NativeMLP
    net = NativeMLP(dims, acts, n_models=n_models)
    if opt is not None:
        net.set_optimizer_kind(opt)
    if w is not None:
        for i in range(n_models):
            net.set_weights(w, model=i)
    return net


def _oracle_fit(w0, acts, X, z, E, perms, l2, l1, opt=None):
    w = [a.copy() for a in w0]
    st = km.AdamState(w) if opt is None else oo.state_for(w, opt)
    h, _ = km.fit(w, acts, X, z, E, 64, perms, adam=st, l2=ro.Factors(l2, l1))
    return h, w


def _close(hist, h_ref, ws, w_ref):
    assert np.abs(hist - h_ref).max() <= LOSS_TOL, np.abs(hist - h_ref).max()
    for a, b in zip(ws, w_ref):
        assert np.abs(a - b).max() <= W_TOL, np.abs(a - b).max()


@pytest.mark.parametrize("mode", [1, 2, 3, 4])
@pytest.mark.parametrize("case", ["l1", "l1_l2", "bias_l1"])
def test_fit_modes(case, mode):
    N, E = 333, 12
    X, z, perms = _problem(DIMS, N, E, seed=5)
    w0 = km.init_weights(DIMS, 3)
    l2, l1 = _factors(case, len(w0))
    h_ref, w_ref = _oracle_fit(w0, ACTS, X, z, E, perms, l2, l1)
    net = _net(DIMS, ACTS, w0)
    net.set_fit_mode(mode)
    hist = net.fit(X, z, E, 64, perms, l2=l2, l1=l1)
    _close(hist, h_ref, net.get_weights(), w_ref)


@pytest.mark.parametrize("mode", [1, 2, 3, 4])
def test_string_through_sequential(mode):
    """``kernel_regularizer="l1_l2"`` (0.01 each) through Sequential.fit and evaluate."""
    from bore_b200.models import Sequential
    N, E = 200, 8
    X, z, perms = _problem(DIMS, N, E, seed=6)
    w0 = km.init_weights(DIMS, 4)
    m = Sequential()
    m.add(layers.Dense(32, activation="elu", input_dim=6, kernel_regularizer="l1_l2", bias_regularizer="l1"))
    m.add(layers.Dense(32, activation="elu", kernel_regularizer="l1_l2", bias_regularizer="l1"))
    m.add(layers.Dense(1, activation="sigmoid"))
    m.compile(optimizer="adam", loss="binary_crossentropy", metrics=["accuracy"])
    m.set_weights(w0)
    m._engine(6).set_fit_mode(mode)
    hist = np.array(m.fit(X, z, batch_size=64, epochs=E, permutations=perms, verbose=0).history["loss"])
    l2 = [0.01, 0.0, 0.01, 0.0, 0.0, 0.0]
    l1 = [0.01, 0.01, 0.01, 0.01, 0.0, 0.0]
    h_ref, w_ref = _oracle_fit(w0, ACTS, X, z, E, perms, l2, l1)
    _close(hist, h_ref, m.get_weights(), w_ref)
    ref = km.evaluate(w_ref, ACTS, X, z, l2=ro.Factors(l2, l1))
    got = m.evaluate(X, z, verbose=0)
    assert abs(got[0] - ref[0]) <= LOSS_TOL and abs(got[1] - ref[1]) <= 1e-6


@pytest.mark.parametrize("dims", [[50, 64, 64, 64, 1], [6, 32, 32, 1], [6, 16, 16, 1], [7, 24, 24, 1],
                                  [7, 40, 40, 1]])
def test_unit_split_builds(dims):
    """Fit mode 4: hidden widths 16 / 32 / 64 take the compile-time builds of the unit-split kernel, 24 / 40 its
    run-time build; the padding of both stays zero under l1."""
    acts = ["tanh"] * (len(dims) - 2) + ["sigmoid"]
    N, E = 700, 4
    X, z, perms = _problem(dims, N, E, seed=9)
    w0 = km.init_weights(dims, 4)
    l2, l1 = _factors("l1_l2", len(w0))
    h_ref, w_ref = _oracle_fit(w0, acts, X, z, E, perms, l2, l1)
    net = _net(dims, acts, w0)
    net.set_fit_mode(4)
    _close(net.fit(X, z, E, 64, perms, l2=l2, l1=l1), h_ref, net.get_weights(), w_ref)


@pytest.mark.parametrize("M", [20, 600])
def test_many_models(M):
    N, E = 150, 6
    probs = [_problem(DIMS, N, E, seed=50 + i) for i in range(M)]
    ws = [km.init_weights(DIMS, 200 + i) for i in range(M)]
    l2, l1 = _factors("l1_l2", len(ws[0]))
    net = _net(DIMS, ACTS, n_models=M)
    for i, w in enumerate(ws):
        net.set_weights(w, model=i)
    net.set_regularizers(l2, l1)
    Xd = net.to_device(np.concatenate([p[0] for p in probs]), np.float32)
    zd = net.to_device(np.concatenate([p[1] for p in probs]).astype(np.float32), np.float32)
    pd = net.to_device(np.stack([p[2] for p in probs]).astype(np.int32), np.int32)
    loss = net.fit_dev(Xd, zd, N, 64, E, pd, model0=0, count=M, shared_data=False, shared_perm=False).cpu().numpy()
    for i in list(range(0, M, max(1, M // 25))) + [M - 1]:
        h_ref, w_ref = _oracle_fit(ws[i], ACTS, probs[i][0], probs[i][1], E, probs[i][2], l2, l1)
        _close(loss[i], h_ref, net.get_weights(model=i), w_ref)


def test_weighted_fit():
    N, E = 200, 10
    X, z, perms = _problem(DIMS, N, E, seed=11)
    sw = np.random.RandomState(12).uniform(0, 2, size=N).astype(np.float32)
    w0 = km.init_weights(DIMS, 6)
    l2, l1 = _factors("l1_l2", len(w0))
    for mode in (1, 2, 3, 4):
        w_ref = [a.copy() for a in w0]
        h_ref, _ = wo.fit(w_ref, ACTS, X, z, E, 64, perms, l2=ro.Factors(l2, l1), sample_weight=sw,
                          class_weight={0: 0.5, 1: 2.0})
        net = _net(DIMS, ACTS, w0)
        net.set_fit_mode(mode)
        hist = net.fit(X, z, E, 64, perms, l2=l2, l1=l1, w=sw, class_weight=(0.5, 2.0))
        _close(hist, h_ref, net.get_weights(), w_ref)


def test_ragged_fit():
    from bore_b200.ragged import RaggedLayout
    n, e = np.array([40, 130, 75]), np.array([9, 3, 5])
    lay = RaggedLayout(n, e)
    probs = [_problem(DIMS, int(n[p]), int(e[p]), seed=20 + p) for p in range(3)]
    ws = [km.init_weights(DIMS, 30 + p) for p in range(3)]
    l2, l1 = _factors("bias_l1", len(ws[0]))
    net = _net(DIMS, ACTS, n_models=3)
    for p, w in enumerate(ws):
        net.set_weights(w, model=p)
    net.set_regularizers(l2, l1)
    Xd = net.to_device(np.concatenate([p[0] for p in probs]), np.float32)
    zd = net.to_device(np.concatenate([p[1] for p in probs]).astype(np.float32), np.float32)
    pd = net.to_device(np.concatenate([p[2].reshape(-1) for p in probs]).astype(np.int32), np.int32)
    loss = net.fit_ragged_dev(Xd, zd, lay, 64, pd).cpu().numpy()
    for p in range(3):
        h_ref, w_ref = _oracle_fit(ws[p], ACTS, probs[p][0], probs[p][1], int(e[p]), probs[p][2], l2, l1)
        _close(loss[lay.losses[p]:lay.losses[p + 1]], h_ref, net.get_weights(model=p), w_ref)


@pytest.mark.parametrize("mode", [1, 2, 3, 4])
def test_extended_activation(mode):
    import activation_oracle as ao
    dims, acts = [6, 32, 32, 1], ["selu", "selu", "sigmoid"]
    N, E = 200, 8
    X, z, perms = _problem(dims, N, E, seed=13)
    w0 = km.init_weights(dims, 7)
    l2, l1 = _factors("l1", len(w0))
    with ao.installed():
        h_ref, w_ref = _oracle_fit(w0, acts, X, z, E, perms, l2, l1)
    net = _net(dims, acts, w0)
    net.set_fit_mode(mode)
    _close(net.fit(X, z, E, 64, perms, l2=l2, l1=l1), h_ref, net.get_weights(), w_ref)


@pytest.mark.parametrize("mode", [1, 2, 3, 4])
@pytest.mark.parametrize("kind", ["nadam", "adagrad"])
def test_other_optimizers(kind, mode):
    o = layers.optimizer_spec(kind)
    N, E = 200, 8
    X, z, perms = _problem(DIMS, N, E, seed=14)
    w0 = km.init_weights(DIMS, 8)
    l2, l1 = _factors("l1_l2", len(w0))
    h_ref, w_ref = _oracle_fit(w0, ACTS, X, z, E, perms, l2, l1, opt=o)
    net = _net(DIMS, ACTS, w0, opt=o)
    net.set_fit_mode(mode)
    _close(net.fit(X, z, E, 64, perms, l2=l2, l1=l1), h_ref, net.get_weights(), w_ref)


@pytest.mark.parametrize("case", ["l1", "l1_l2", "bias_l1"])
def test_evaluate(case):
    """Plain and weighted evaluate carry the l1 penalty; a trained net, so no parameter sits at zero."""
    N = 300
    X, z, perms = _problem(DIMS, N, 4, seed=15)
    w0 = km.init_weights(DIMS, 9)
    l2, l1 = _factors(case, len(w0))
    net = _net(DIMS, ACTS, w0)
    net.fit(X, z, 4, 64, perms)
    w = [np.asarray(a) for a in net.get_weights()]
    got = net.evaluate(X, z, l2=l2, l1=l1)
    ref = km.evaluate(w, ACTS, X, z, l2=ro.Factors(l2, l1))
    assert abs(got[0] - ref[0]) <= 1e-5 and abs(got[1] - ref[1]) <= 1e-6
    assert got[0] - net.evaluate(X, z, l2=l2)[0] >= 0.5 * ro.l1_penalty(w, l1)  # the l1 term is there
    sw = np.random.RandomState(16).uniform(0, 2, size=N).astype(np.float32)
    got = net.evaluate(X, z, l2=l2, l1=l1, w=sw, class_weight=(0.5, 2.0))
    ref = wo.evaluate(w, ACTS, X, z, l2=ro.Factors(l2, l1), sample_weight=sw, class_weight={0: 0.5, 1: 2.0})
    assert abs(got[0] - ref[0]) <= 1e-5 and abs(got[1] - ref[1]) <= 1e-6


def _lstm_factors(L):
    """The factors of the factory below: l1_l2 on the kernels, "l1" (0.01) on the recurrent kernels, l1 on the biases
    and on both arrays of the final layer."""
    n = 3 * L + 2
    l1 = [(1e-3, 0.01, 3e-3)[i % 3] for i in range(3 * L)] + [2e-3, 4e-3]
    l2 = [1e-3 if i % 3 == 0 else 0.0 for i in range(3 * L)] + [0.0, 0.0]
    assert len(l1) == len(l2) == n
    return l2, l1


def test_lstm_fit_and_evaluate():
    from bore_b200.layers import BinaryCrossentropy
    from bore_b200.models import StackedRecurrentFactory
    D, U, L, N, B, T, mv, E = 8, 32, 2, 100, 64, 4, -1.0, 12
    X, Y = lstm_sequences(4, N, T, D, mv)
    rs = np.random.RandomState(5)
    perms = np.stack([rs.permutation(N) for _ in range(E)])
    w0 = kl.init_weights(D, U, L, seed=6)
    l2, l1 = _lstm_factors(L)
    w64 = [a.astype(np.float64) for a in w0]
    h64, _ = kl.fit(w64, "tanh", X, Y, E, B, perms, mv, adam=km.AdamState(w64), l2=ro.Factors(l2, l1),
                    dtype=np.float64)
    fac = StackedRecurrentFactory(D, 1, num_layers=L, num_units=U, seed=0,
                                  layer_kws=dict(activation="tanh", kernel_regularizer=layers.L1L2(1e-3, 1e-3),
                                                 recurrent_regularizer="l1",
                                                 bias_regularizer=layers.l1(3e-3)),
                                  final_layer_kws=dict(kernel_regularizer=layers.L1(2e-3),
                                                       bias_regularizer=layers.L1(4e-3)))
    assert fac._factors() == (l2, l1)
    net = fac.build_many_to_many(mask_value=mv)
    net.compile(optimizer="adam", loss=BinaryCrossentropy(from_logits=True))
    net.set_weights(w0)
    hist = np.array(net.fit(X, Y, epochs=E, batch_size=B, permutations=perms, verbose=0).history["loss"])
    assert np.abs(hist - h64).max() <= LOSS_TOL, (hist, h64)
    for a, b in zip(net.get_weights(), w64):
        assert np.abs(a - b).max() <= W_TOL
    w = [np.asarray(a, np.float64) for a in net.get_weights()]
    got = net.evaluate(X, Y)
    ref = ro.lstm_evaluate(w, "tanh", X, Y, mv, ro.Factors(l2, l1), dtype=np.float64)
    assert abs(got - ref[0]) <= 1e-5, (got, ref)


def test_batched_surface():
    """BatchedMaximizableSequential compiled with l1 layers: every problem follows its own oracle fit."""
    from bore_b200 import BatchedMaximizableSequential, Dense
    M, D, N, E = 5, 4, 80, 6
    model = BatchedMaximizableSequential([Dense(16, activation="relu", input_dim=D, kernel_regularizer="l1",
                                                bias_regularizer=layers.l1_l2(1e-3, 2e-3)),
                                          Dense(16, activation="relu", kernel_regularizer=layers.L1L2(l1=5e-3)),
                                          Dense(1, activation="sigmoid")], n_problems=M, seed=2)
    model.compile(optimizer="adam", loss="binary_crossentropy")
    dims, acts = [D, 16, 16, 1], ["relu", "relu", "sigmoid"]
    ws = [km.init_weights(dims, 40 + p) for p in range(M)]
    model.set_weights(ws)
    rs = np.random.RandomState(1)
    X = rs.uniform(size=(M, N, D))
    y = np.sum((X - 0.4) ** 2, axis=2)
    z = (y < np.quantile(y, 0.3, axis=1, keepdims=True)).astype(np.float32)
    perms = np.stack([np.stack([rs.permutation(N) for _ in range(E)]) for _ in range(M)])
    loss = np.asarray(model.fit(X, z, batch_size=32, epochs=E, permutations=perms))
    l2 = [0.0, 2e-3, 0.0, 0.0, 0.0, 0.0]
    l1 = [0.01, 1e-3, 5e-3, 0.0, 0.0, 0.0]
    for p in range(M):
        w = [a.copy() for a in ws[p]]
        h_ref, _ = km.fit(w, acts, X[p], z[p], E, 32, perms[p], adam=km.AdamState(w), l2=ro.Factors(l2, l1))
        _close(loss[p], h_ref, model.get_weights()[p], w)


def test_zero_l1_is_bit_identical():
    """set_regularizers(l2, l1=zeros) runs exactly what set_regularizers(l2) runs: every fit mode and the LSTM."""
    N, E = 200, 5
    X, z, perms = _problem(DIMS, N, E, seed=17)
    w0 = km.init_weights(DIMS, 11)
    l2 = [1e-3, 0.0, 1e-3, 0.0, 0.0, 0.0]
    for mode in (1, 2, 3, 4):
        out = []
        for l1 in (None, [0.0] * 6):
            net = _net(DIMS, ACTS, w0)
            net.set_fit_mode(mode)
            net.set_regularizers(l2, l1)
            out.append((net.fit(X, z, E, 64, perms), net.get_weights(), net.get_optimizer_state(),
                        net.evaluate(X, z)))
        (ha, wa, sa, ea), (hb, wb, sb, eb) = out
        assert np.array_equal(ha, hb) and ea == eb, mode
        assert all(np.array_equal(a, b) for a, b in zip(wa, wb)), mode
        assert all(np.array_equal(a, b) for a, b in zip(sa[0] + sa[1], sb[0] + sb[1])) and sa[2] == sb[2], mode
    D, U, L, T, mv = 8, 32, 2, 4, -1.0
    Xs, Ys = lstm_sequences(4, 64, T, D, mv)
    out = []
    for l1 in (None, [0.0] * (3 * L + 2)):
        net = lstm_factory(D, U, L, "tanh")._engine()
        net.set_weights(kl.init_weights(D, U, L, seed=6))
        net.set_regularizers([1e-3] * (3 * L + 2), l1)
        loss = net.fit_async(Xs, Ys, 3, 32, np.stack([np.arange(64)] * 3), mv).cpu().numpy()
        out.append((loss, net.get_weights(), net.get_adam_state(), net.evaluate(Xs, Ys, mv)))
    (ha, wa, sa, ea), (hb, wb, sb, eb) = out
    assert np.array_equal(ha, hb) and list(ea) == list(eb)
    assert all(np.array_equal(a, b) for a, b in zip(wa, wb))
    assert all(np.array_equal(a, b) for a, b in zip(list(sa[0]) + list(sa[1]), list(sb[0]) + list(sb[1])))
    assert sa[2] == sb[2]


@pytest.mark.parametrize("mode", [1, 2, 3, 4])
def test_zero_bias_gets_no_l1_gradient(mode):
    """One step from zero biases under bias-only l1 moves every parameter exactly as with no regulariser.  Nadam, so
    that both runs take the same build of every kernel: the one-CTA kernel's Adam build has no l1 terms, and a fit
    with l1 runs its other build."""
    N = 64
    X, z, perms = _problem(DIMS, N, 1, seed=18)
    w0 = km.init_weights(DIMS, 12)
    assert not any(w0[i].any() for i in (1, 3, 5))
    got = []
    for l1 in (None, [0.0, 0.5, 0.0, 0.5, 0.0, 0.5]):
        net = _net(DIMS, ACTS, w0, opt=layers.Nadam())
        net.set_fit_mode(mode)
        net.set_regularizers(0.0, l1)
        got.append((net.fit(X, z, 1, 64, perms), net.get_weights()))
    assert np.array_equal(got[0][0], got[1][0])
    for a, b in zip(got[0][1], got[1][1]):
        assert np.array_equal(a, b)


def test_native_argument_checks(native_lib):
    lib = native_lib
    net = _net(DIMS, ACTS)
    lstm = lstm_factory(8, 16, 2, "tanh")._engine()
    ok = (C.c_float * 8)(*([1e-3] * 8))
    for bad in (-1e-3, float("nan"), float("inf")):
        arr = (C.c_float * 8)(*([1e-3] * 7 + [bad]))
        assert lib.bore_lstm_set_l1_regularizers(lstm.h, arr) != 0
        assert "must be finite and >= 0" in lib.bore_last_error().decode()
        k = (C.c_float * 3)(1e-3, bad, 0.0)
        assert lib.bore_mlp_set_l1_regularizers(net.h, k, ok) != 0
        assert "must be finite and >= 0" in lib.bore_last_error().decode()
        assert lib.bore_mlp_set_l1_regularizers(net.h, ok, k) != 0
    assert lib.bore_mlp_set_l1_regularizers(None, ok, ok) != 0
    assert "NULL" in lib.bore_last_error().decode()
    assert lib.bore_lstm_set_l1_regularizers(None, ok) != 0
    assert "NULL" in lib.bore_last_error().decode()
    assert lib.bore_mlp_set_l1_regularizers(net.h, ok, ok) == 0
    assert lib.bore_lstm_set_l1_regularizers(lstm.h, ok) == 0
    with pytest.raises(RuntimeError, match="must be finite and >= 0"):
        net.set_regularizers(0.0, [1e-3, -1.0, 0, 0, 0, 0])
