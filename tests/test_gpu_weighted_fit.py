"""Weighted training (Keras ``sample_weight`` / ``class_weight``) on the GPU: every fit kernel against
the oracle, the exact properties of the weighting (unit weights are the unweighted fit bit for bit,
zero-weight samples do not matter), many models per launch, the batched surface with labels made on
the device, and ``evaluate``."""
import functools

import numpy as np
import pytest

from oracle import keras_mlp as km
import weighted_oracle as wo
from helpers import NETS, synthetic_targets

pytestmark = pytest.mark.gpu

# the net-shape envelope's own cases (copied from test_gpu_shapes.py): a weighted fit must take exactly
# the (net, mode, batch) cases an unweighted one takes, and refuse the others with the same error
SHAPES = {
    "odd": ([5, 3, 17, 1], ["elu", "tanh", "sigmoid"]),
    "w65": ([9, 65, 63, 1], ["relu", "elu", "sigmoid"]),
    "deep7_mixed": ([10, 16, 48, 8, 96, 24, 64, 40, 1],
                    ["tanh", "relu", "elu", "sigmoid", "relu", "linear", "elu", "sigmoid"]),
    "edge_32x2": ([465, 32, 32, 1], ["tanh", "tanh", "sigmoid"]),
    "edge_64x3": ([139, 64, 64, 64, 1], ["elu", "elu", "elu", "sigmoid"]),
    "edge_128x1": ([156, 128, 1], ["tanh", "sigmoid"]),
}
for _n, (_d, _a, _) in NETS.items():
    SHAPES[_n] = (_d, list(_a))

_UNIT = "unit-split cluster kernel does not take"
_MMA = "tensor-pipe kernel does not take"
FIT_REFUSED = {
    ("deep7_mixed", 4, 64): _UNIT, ("d512", 4, 64): _UNIT, ("nohid300", 4, 64): _UNIT,
    ("edge_32x2", 4, 64): _UNIT, ("edge_64x3", 4, 64): _UNIT, ("edge_128x1", 4, 64): _UNIT,
    ("edge_32x2", 2, 64): "cluster mode needs 285328 B",
    ("edge_64x3", 2, 64): "cluster mode needs 301680 B",
    ("edge_128x1", 2, 64): "cluster mode needs 301776 B",
    ("odd", 4, 100): _UNIT, ("odd", 4, 128): _UNIT, ("w65", 4, 100): _UNIT, ("w65", 4, 128): _UNIT,
    ("deep7_mixed", 4, 100): _UNIT, ("deep7_mixed", 4, 128): _UNIT,
    ("deep7_mixed", 1, 100): "model \\+ batch of 100 need 282896 B",
    ("deep7_mixed", 1, 128): "model \\+ batch of 128 need 339008 B",
    ("deep7_mixed", 3, 64): _MMA,
}
LOSS_TOL = 1e-4
EPOCHS = 6

# weightings: (sample weights, class weights) as the engine takes them
KINDS = ("positive", "zeros", "class", "both")


def _weighting(kind, z, seed):
    rs = np.random.RandomState(seed)
    n = len(z)
    w = None
    if kind in ("positive", "both"):
        w = rs.uniform(0.25, 2.0, size=n).astype(np.float32)
    if kind == "zeros":
        w = rs.uniform(0.5, 1.5, size=n).astype(np.float32)
        w[rs.uniform(size=n) < 0.3] = 0.0
    cw = (0.5, 2.0) if kind in ("class", "both") else None
    return w, cw


def _oracle_kwargs(w, cw):
    return dict(sample_weight=w, class_weight=None if cw is None else {0: cw[0], 1: cw[1]})


def _problem(dims, N, epochs, seed):
    rs = np.random.RandomState(seed)
    X = rs.uniform(size=(N, dims[0]))
    y = synthetic_targets(X)
    z = y < np.quantile(y, 0.25)
    perms = np.stack([rs.permutation(N) for _ in range(epochs)])
    return X, z, perms


@functools.lru_cache(maxsize=None)
def _case(name, batch, kind):
    dims, acts = SHAPES[name]
    N = 40 if batch < 8 else 150
    X, z, perms = _problem(dims, N, EPOCHS, seed=batch + dims[0])
    w, cw = _weighting(kind, z, seed=batch + 7)
    w0 = km.init_weights(dims, 3)
    w_ref = [a.copy() for a in w0]
    hist_ref, adam_ref = wo.fit(w_ref, acts, X, z, EPOCHS, batch, perms, **_oracle_kwargs(w, cw))
    return X, z, perms, w, cw, w0, hist_ref, w_ref, adam_ref


def _assert_matches(net, hist, case, batch):
    X, z, perms, w, cw, w0, hist_ref, w_ref, adam_ref = case
    assert np.abs(hist - hist_ref).max() <= LOSS_TOL, np.abs(hist - hist_ref).max()
    for a, b in zip(net.get_weights(), w_ref):
        assert np.abs(a - b).max() <= 2e-3, np.abs(a - b).max()
    m, v, t = net.get_adam_state()
    assert t == adam_ref.t == EPOCHS * (-(-len(X) // batch))
    for a, b in zip(m, adam_ref.m):
        assert np.abs(a - b).max() <= 1e-4


CASES = [(n, m, 64) for n in SHAPES for m in (1, 2, 3, 4)]
CASES += [(n, m, b) for n in ("odd", "w65", "deep7_mixed") for m in (1, 2, 4) for b in (1, 5, 100, 128)]


@pytest.mark.parametrize("name,mode,batch", CASES)
def test_weighted_fit_matches_oracle(name, mode, batch):
    """Every net x mode x batch: the weighted fit is taken where the unweighted one is (and refused with
    the same error where it is not), and then matches the weighted oracle.  The weighting rotates over
    positive weights, weights with zeros, class weights alone, and both."""
    from bore_b200.engine import NativeMLP
    from bore_b200._lib import BoreNativeError
    dims, acts = SHAPES[name]
    kind = KINDS[(CASES.index((name, mode, batch))) % len(KINDS)]
    case = _case(name, batch, kind)
    X, z, perms, w, cw, w0 = case[:6]
    net = NativeMLP(dims, acts)
    net.set_fit_mode(mode)
    net.set_weights(w0)
    try:
        net.fit(X, z, EPOCHS, batch, perms)
        unweighted_error = None
    except BoreNativeError as e:
        unweighted_error = str(e)
    refused = FIT_REFUSED.get((name, mode, batch))
    if refused:
        assert unweighted_error is not None
    if unweighted_error is not None:
        with pytest.raises(BoreNativeError) as info:
            net.fit(X, z, EPOCHS, batch, perms, w=w, class_weight=cw)
        assert str(info.value) == unweighted_error
        return
    net = NativeMLP(dims, acts)
    net.set_fit_mode(mode)
    net.set_weights(w0)
    hist = net.fit(X, z, EPOCHS, batch, perms, w=w, class_weight=cw)
    _assert_matches(net, hist, case, batch)


def _run(dims, acts, mode, w0, X, z, perms, batch, **kw):
    from bore_b200.engine import NativeMLP
    net = NativeMLP(dims, acts)
    net.set_fit_mode(mode)
    net.set_weights(w0)
    hist = net.fit(X, z, EPOCHS, batch, perms, **kw)
    return hist, net.get_weights(), net.get_adam_state()


def _assert_identical(a, b):
    ha, wa, (ma, va, ta) = a
    hb, wb, (mb, vb, tb) = b
    assert np.array_equal(ha, hb)
    assert ta == tb
    for x, y in zip(wa + ma + va, wb + mb + vb):
        assert np.array_equal(x, y)


# cfg3 is a compile-time K1u build (3 x 64, batch 64), "odd" the run-time-shape build
@pytest.mark.parametrize("name", ["cfg3_ackley50", "odd"])
@pytest.mark.parametrize("mode", [1, 2, 3, 4])
def test_unit_weights_are_the_unweighted_fit_bit_for_bit(name, mode):
    dims, acts = SHAPES[name]
    X, z, perms = _problem(dims, 150, EPOCHS, seed=4)
    w0 = km.init_weights(dims, 5)
    ref = _run(dims, acts, mode, w0, X, z, perms, 64)
    ones = np.ones(len(X), np.float32)
    _assert_identical(ref, _run(dims, acts, mode, w0, X, z, perms, 64, w=ones, class_weight=(1.0, 1.0)))
    _assert_identical(ref, _run(dims, acts, mode, w0, X, z, perms, 64, w=ones))
    _assert_identical(ref, _run(dims, acts, mode, w0, X, z, perms, 64, class_weight=(1.0, 1.0)))


@pytest.mark.parametrize("name", ["cfg2_hartmann6", "odd"])
@pytest.mark.parametrize("mode", [1, 2, 3, 4])
def test_labels_of_zero_weight_samples_do_not_matter(name, mode):
    dims, acts = SHAPES[name]
    X, z, perms = _problem(dims, 150, EPOCHS, seed=6)
    w, _ = _weighting("zeros", z, seed=1)
    w0 = km.init_weights(dims, 6)
    flipped = np.where(w == 0, ~z, z)
    assert (flipped != z).sum() > 10
    a = _run(dims, acts, mode, w0, X, z, perms, 64, w=w, class_weight=(0.7, 1.3))
    b = _run(dims, acts, mode, w0, X, flipped, perms, 64, w=w, class_weight=(0.7, 1.3))
    _assert_identical(a, b)


# ---------------------------------------------------------------- many models, one CTA each
@pytest.mark.parametrize("M", [20, 600])
@pytest.mark.parametrize("shared", [False, True])
def test_many_models_weighted(M, shared):
    from bore_b200.engine import NativeMLP
    dims, acts = SHAPES["w65"] if M == 20 else SHAPES["cfg2_hartmann6"]
    N, E = 150, EPOCHS
    probs = [_problem(dims, N, E, seed=50 + (0 if shared else i)) for i in range(M)]
    wts = [_weighting("zeros" if i % 2 else "positive", probs[i][1], seed=i)[0] for i in range(M)]
    cw = (0.6, 1.8)
    ws = [km.init_weights(dims, 200 + i) for i in range(M)]
    net = NativeMLP(dims, acts, n_models=M)
    for i, w in enumerate(ws):
        net.set_weights(w, model=i)
    k = 1 if shared else M
    Xd = net.to_device(np.concatenate([p[0] for p in probs[:k]]), np.float32)
    zd = net.to_device(np.concatenate([p[1] for p in probs[:k]]).astype(np.float32), np.float32)
    wd = net.to_device(np.concatenate(wts[:k]), np.float32)
    pd = net.to_device(np.stack([p[2] for p in probs]).astype(np.int32), np.int32)
    loss = net.fit_dev(Xd, zd, N, 64, E, pd, model0=0, count=M, shared_data=shared, shared_perm=False,
                       w_dev=wd, class_weight=cw).cpu().numpy()
    for i in range(M):
        j = 0 if shared else i
        w_ref = [a.copy() for a in ws[i]]
        h_ref, _ = wo.fit(w_ref, acts, probs[j][0], probs[j][1], E, 64, probs[i][2],
                          **_oracle_kwargs(wts[j], cw))
        assert np.abs(loss[i] - h_ref).max() <= LOSS_TOL, (i, np.abs(loss[i] - h_ref).max())
        for u, v in zip(net.get_weights(model=i), w_ref):
            assert np.abs(u - v).max() <= 2e-3, i


def test_batched_weighted_fit_with_device_labels():
    """64 cfg-2-shaped problems, labels z = y < quantile(y, gamma) made on the device, class weights
    applied there; the oracle gets the host's quantile labels."""
    from bore_b200 import BatchedMaximizableSequential, Dense
    M, N, D, E, gamma = 64, 100, 6, 6, 0.25
    dims, acts = [D, 32, 32, 1], ["relu", "relu", "sigmoid"]
    rs = np.random.RandomState(9)
    X = rs.uniform(size=(M, N, D))
    y = np.stack([synthetic_targets(X[p]) + 0.2 * p * X[p, :, 1] for p in range(M)])
    sw = rs.uniform(0.0, 2.0, size=(M, N)).astype(np.float32)
    cw = {0: 0.4, 1: 3.0}
    layers = [Dense(32, activation="relu", input_dim=D), Dense(32, activation="relu"),
              Dense(1, activation="sigmoid")]
    model = BatchedMaximizableSequential(layers, n_problems=M, seed=3)
    model.compile(optimizer="adam", loss="binary_crossentropy")
    w0 = model.get_weights()
    perms = np.stack([np.stack([rs.permutation(N) for _ in range(E)]) for _ in range(M)])
    hist = np.asarray(model.fit(X, y, batch_size=32, epochs=E, permutations=perms, gamma=gamma,
                                sample_weight=sw, class_weight=cw))
    got = model.get_weights()
    for p in range(M):
        z = y[p] < np.quantile(y[p], gamma)
        w = [a.copy() for a in w0[p]]
        h_ref, _ = wo.fit(w, acts, X[p], z, E, 32, perms[p], sample_weight=sw[p], class_weight=cw)
        assert np.abs(hist[p] - h_ref).max() <= LOSS_TOL, p
        for a, b in zip(got[p], w):
            assert np.abs(a - b).max() <= 2e-3, p
    with pytest.raises(ValueError):
        model.fit(X, y, batch_size=32, epochs=1, gamma=gamma, class_weight={0: 1.0})
    with pytest.raises(ValueError):
        model.fit(X, y, batch_size=32, epochs=1, gamma=gamma, sample_weight=np.ones((M, N + 1)))


# ---------------------------------------------------------------- the model surface
def _model(dims, acts, seed=0):
    from bore_b200.models import MaximizableSequential
    from bore_b200.layers import Dense
    model = MaximizableSequential(seed=seed)
    for i, (u, a) in enumerate(zip(dims[1:], acts)):
        model.add(Dense(u, activation=a, input_dim=dims[0] if i == 0 else None))
    return model


def test_sequential_weighted_fit_then_argmax():
    from scipy.optimize import Bounds
    dims, acts = SHAPES["cfg2_hartmann6"]
    X, z, perms = _problem(dims, 120, 8, seed=11)
    sw = np.random.RandomState(2).uniform(0.0, 2.0, size=(120, 1))
    model = _model(dims, acts)
    model.compile(optimizer="adam", loss="binary_crossentropy", metrics=["accuracy"])
    w0 = model.get_weights()
    hist = model.fit(X, z, batch_size=32, epochs=8, verbose=0, permutations=perms, sample_weight=sw,
                     class_weight={0: 1.0, 1: 3.0})
    w_ref = [a.copy() for a in w0]
    h_ref, _ = wo.fit(w_ref, acts, X, z, 8, 32, perms, sample_weight=sw, class_weight={0: 1.0, 1: 3.0})
    assert np.abs(np.array(hist.history["loss"]) - h_ref).max() <= LOSS_TOL
    res = model.argmax(Bounds(np.zeros(6), np.ones(6)), num_starts=4, num_samples=256, print_fn=None,
                       random_state=np.random.RandomState(0))
    assert res is not None and np.all(res.x >= 0) and np.all(res.x <= 1)
    with pytest.raises(ValueError):
        model.fit(X, z, epochs=1, verbose=0, class_weight={1: 1.0, 2: 1.0})
    with pytest.raises(ValueError):
        model.fit(X, z, epochs=1, verbose=0, sample_weight=np.ones(119))


@pytest.mark.parametrize("name", ["cfg2_hartmann6", "cfg5_plugin8", "tanh_exp"])
def test_weighted_evaluate_matches_oracle(name):
    dims, acts = SHAPES[name]
    from helpers import trained_weights
    w = trained_weights(dims, acts, seed=2, N=150, epochs=6)
    model = _model(dims, acts)
    from bore_b200.layers import BinaryCrossentropy
    loss = "binary_crossentropy" if acts[-1] == "sigmoid" else BinaryCrossentropy(from_logits=True)
    model.compile(optimizer="adam", loss=loss, metrics=["accuracy"])
    model.set_weights(w)
    rs = np.random.RandomState(1)
    X = rs.uniform(size=(333, dims[0]))
    z = synthetic_targets(X) < 0.5
    for sw in (rs.uniform(0.0, 2.0, size=333), np.where(rs.uniform(size=333) < 0.5, 0.0, 1.5),
               np.zeros(333), np.ones((333, 1))):
        got = model.evaluate(X, z, sample_weight=sw)
        ref = wo.evaluate(model.get_weights(), acts, X, z, sample_weight=sw)
        assert abs(got[0] - ref[0]) <= 1e-5 and abs(got[1] - ref[1]) <= 1e-6, (got, ref)
    # class weights through the engine
    got = model._engine().evaluate(X, z, w=np.ones(333), class_weight=(0.5, 2.0))
    ref = wo.evaluate(model.get_weights(), acts, X, z, sample_weight=np.ones(333), class_weight={0: 0.5, 1: 2.0})
    assert abs(got[0] - ref[0]) <= 1e-5 and abs(got[1] - ref[1]) <= 1e-6, (got, ref)
