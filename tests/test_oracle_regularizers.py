"""Keras l1 and l1_l2 regularisation: the oracle's rule (tests/regularizer_oracle.py) against an independent torch-CPU
autograd implementation in fp64 (torch's ``abs`` backward is ``sign``, 0 at 0, as TF's), and the host-side surface
(classes, defaults, ``regularizer_get``, refusals, the header).  CPU only."""
import os
import re

import numpy as np
import pytest
import torch

from oracle import keras_lstm as kl, keras_mlp as km
import regularizer_oracle as ro
from bore_b200 import layers
from bore_b200.models import Sequential, StackedRecurrentFactory
from test_oracle_optimizers import _Hand, _torch_lstm, _torch_mlp

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _factors(case, n):
    """Per-array (l2, l1) factors of a case, Keras order [k0, b0, k1, b1, ...]."""
    if case == "l1":
        return [0.0] * n, [1e-3] * n
    if case == "l1_l2":
        return [1e-3] * n, [2e-3] * n
    assert case == "bias_l1"
    return [0.0] * n, [0.0 if i % 2 == 0 else 5e-3 for i in range(n)]


def _torch_fit(w0, loss_fn, N, epochs, batch, perms, l2, l1):
    ws = [torch.tensor(a, requires_grad=True) for a in w0]
    opt = _Hand(ws, layers.Adam(learning_rate=5e-3))
    hist = []
    for e in range(epochs):
        tot = 0.0
        for s in range(0, N, batch):
            idx = torch.as_tensor(perms[e][s:s + batch])
            loss = loss_fn(ws, idx)
            loss = loss + sum(f1 * a.abs().sum() + f2 * (a * a).sum() for a, f2, f1 in zip(ws, l2, l1))
            opt.zero_grad()
            loss.backward()
            opt.step()
            tot += float(loss.detach()) * len(idx)
        hist.append(tot / N)
    return np.array(hist), [a.detach().numpy() for a in ws]


@pytest.mark.parametrize("case", ["l1", "l1_l2", "bias_l1"])
@pytest.mark.parametrize("dims,acts", [([4, 16, 8, 1], ["elu", "tanh", "sigmoid"]), ([3, 12, 1], ["relu", "linear"])])
def test_mlp_fit_vs_torch(case, dims, acts):
    """100 steps (25 epochs x 4 batches) of the oracle fit loop with the l1 rule."""
    rs = np.random.RandomState(3)
    N, E, B = 100, 25, 25
    X = rs.uniform(-1.5, 1.5, size=(N, dims[0]))
    y = np.sum((X - 0.3) ** 2, axis=1)
    z = (y < np.quantile(y, 0.3)).astype(np.float64)
    perms = np.stack([rs.permutation(N) for _ in range(E)])
    w0 = km.init_weights(dims, 5, np.float64)
    w = [a.copy() for a in w0]
    l2, l1 = _factors(case, len(w0))
    with ro.installed():
        hist, st = km.fit(w, acts, X, z, E, B, perms, adam=km.AdamState(w, lr=5e-3), l2=ro.Factors(l2, l1),
                          dtype=np.float64)
    assert st.t == 100
    Xt, zt = torch.tensor(X), torch.tensor(z).reshape(-1, 1)
    bce = torch.nn.functional.binary_cross_entropy_with_logits
    hist_t, wt = _torch_fit(w0, lambda ws, idx: bce(_torch_mlp(ws, acts, Xt[idx]), zt[idx]), N, E, B, perms, l2, l1)
    assert np.abs(hist - hist_t).max() <= 1e-10
    assert max(np.abs(a - b).max() for a, b in zip(w, wt)) <= 1e-10
    # the l1 terms changed the result: the same fit without them ends elsewhere
    w_plain = [a.copy() for a in w0]
    km.fit(w_plain, acts, X, z, E, B, perms, adam=km.AdamState(w_plain, lr=5e-3), l2=l2, dtype=np.float64)
    assert max(np.abs(a - b).max() for a, b in zip(w, w_plain)) > 1e-6


@pytest.mark.parametrize("case", ["l1", "l1_l2", "bias_l1"])
def test_lstm_fit_vs_torch(case):
    """100 steps (50 epochs x 2 batches) of keras_lstm's fit loop with the l1 rule on every array kind."""
    D, U, L, T, N, E, B = 4, 8, 2, 3, 40, 50, 20
    rs = np.random.RandomState(7)
    X = rs.uniform(size=(N, T, D))
    Y = (rs.uniform(size=(N, T, 1)) < 0.4).astype(np.float64)
    perms = np.stack([rs.permutation(N) for _ in range(E)])
    w0 = kl.init_weights(D, U, L, seed=8, dtype=np.float64)
    w = [a.copy() for a in w0]
    l2, l1 = _factors(case, len(w0))
    if case == "bias_l1":  # Keras order per cell: kernel, recurrent kernel, bias; then the Dense kernel and bias
        l1 = [5e-3 if (i < 3 * L and i % 3 == 2) or i == 3 * L + 1 else 0.0 for i in range(len(w0))]
    with ro.installed():
        hist, st = kl.fit(w, "tanh", X, Y, E, B, perms, mask_value=-1e9, adam=km.AdamState(w, lr=5e-3),
                          l2=ro.Factors(l2, l1), dtype=np.float64)
    assert st.t == 100
    Xt, Yt = torch.tensor(X), torch.tensor(Y[..., 0])
    bce = torch.nn.functional.binary_cross_entropy_with_logits
    hist_t, wt = _torch_fit(w0, lambda ws, idx: bce(_torch_lstm(ws, Xt[idx]), Yt[idx]), N, E, B, perms, l2, l1)
    assert np.abs(hist - hist_t).max() <= 1e-10
    assert max(np.abs(a - b).max() for a, b in zip(w, wt)) <= 1e-10


def test_evaluate_losses_carry_l1():
    """MLP and LSTM evaluate: the loss is the data loss plus l1 sum|w| + l2 sum w^2."""
    rs = np.random.RandomState(0)
    w = km.init_weights([3, 8, 1], 1, np.float64)
    w[1] = rs.normal(size=w[1].shape)
    X, z = rs.normal(size=(20, 3)), (rs.uniform(size=20) < 0.5).astype(np.float64)
    l2, l1 = _factors("l1_l2", len(w))
    plain = km.evaluate(w, ["relu", "sigmoid"], X, z, dtype=np.float64)[0]
    with ro.installed():
        got = km.evaluate(w, ["relu", "sigmoid"], X, z, l2=ro.Factors(l2, l1), dtype=np.float64)[0]
    want = plain + sum(f2 * np.sum(a * a) + f1 * np.sum(np.abs(a)) for a, f2, f1 in zip(w, l2, l1))
    assert abs(got - want) <= 1e-12
    wl = kl.init_weights(3, 4, 1, seed=2, dtype=np.float64)
    Xs, Ys = rs.uniform(size=(6, 2, 3)), (rs.uniform(size=(6, 2, 1)) < 0.5).astype(np.float64)
    l2, l1 = _factors("l1", len(wl))
    got = ro.lstm_evaluate(wl, "tanh", Xs, Ys, -1e9, ro.Factors(l2, l1), dtype=np.float64)[0]
    want = kl.evaluate(wl, "tanh", Xs, Ys, -1e9, dtype=np.float64)[0] + 1e-3 * sum(np.abs(a).sum() for a in wl)
    assert abs(got - want) <= 1e-12


def test_zero_parameter_gets_no_l1_gradient():
    """sign(0) = 0: a zero array under l1 keeps the gradient it has without a regulariser."""
    w = km.init_weights([3, 4, 1], 0, np.float64)
    assert not w[1].any()  # biases start at zero
    X, z = np.ones((5, 3)), np.array([0, 1, 0, 1, 1], np.float64)
    _, g0 = km.loss_and_weight_grads(w, ["relu", "sigmoid"], X, z, 0.0, np.float64)
    with ro.installed():
        _, g1 = km.loss_and_weight_grads(w, ["relu", "sigmoid"], X, z, ro.Factors(0.0, [0, 1.0, 0, 1.0]),
                                         np.float64)
    assert np.array_equal(g0[1], g1[1]) and np.array_equal(g0[3], g1[3])


def test_installed_restores_the_oracle():
    with ro.installed():
        assert km.loss_and_weight_grads is not ro._KM_LOSS
    assert km.loss_and_weight_grads is ro._KM_LOSS and kl.loss_and_weight_grads is ro._KL_LOSS


def test_classes_and_defaults():
    assert layers.L1().l1 == 0.01 and layers.l1 is layers.L1 and layers.l1(0.5).l1 == 0.5
    assert layers.L2().l2 == 0.01 and layers.l2(0.2).l2 == 0.2
    c = layers.L1L2()
    assert (c.l1, c.l2) == (0.0, 0.0)
    c = layers.l1_l2()
    assert isinstance(c, layers.L1L2) and (c.l1, c.l2) == (0.01, 0.01)
    c = layers.l1_l2(l1=0.1)
    assert (c.l1, c.l2) == (0.1, 0.01)
    assert layers.regularizer_factors([None, layers.L1(0.5), layers.L2(0.25), layers.L1L2(0.125, 2.0)]) == \
        ([0.0, 0.0, 0.25, 2.0], [0.0, 0.5, 0.0, 0.125])


def test_regularizer_get():
    get = layers.regularizer_get
    assert get(None, "x") is None
    inst = layers.L1(0.3)
    assert get(inst, "x") is inst
    for name, cls in (("l1", layers.L1), ("L1", layers.L1), ("l2", layers.L2), ("L2", layers.L2)):
        r = get(name, "x")
        assert type(r) is cls and getattr(r, name.lower()) == 0.01
    r = get("L1L2", "x")  # the class: zeros
    assert type(r) is layers.L1L2 and (r.l1, r.l2) == (0.0, 0.0)
    r = get("l1_l2", "x")  # deserialize's special case: 0.01 each
    assert type(r) is layers.L1L2 and (r.l1, r.l2) == (0.01, 0.01)


def test_refusals_at_construction():
    class Own:
        l2 = 0.1

    for bad in ("l3", "L1_L2", "l1l2", Own(), lambda w: 0.0, 0.01, {"class_name": "L1"}):
        with pytest.raises(ValueError, match="must be None, an instance of bore_b200.layers.{L1, L2, L1L2}"):
            layers.Dense(4, kernel_regularizer=bad)
        with pytest.raises(ValueError, match="LSTMCell"):
            from bore_b200.recurrent import LSTMCell
            LSTMCell(4, recurrent_regularizer=bad)
    with pytest.raises(ValueError, match="Dense"):
        layers.Dense(4, bias_regularizer="l3")
    for bad in (-1e-3, float("nan"), float("inf")):
        with pytest.raises(ValueError, match="finite and >= 0"):
            layers.L1(bad)
        with pytest.raises(ValueError, match="finite and >= 0"):
            layers.L1L2(l2=bad)


def test_surfaces_resolve_strings():
    """Sequential and the recurrent factory turn every accepted form into the factors they send to the kernels."""
    m = Sequential()
    m.add(layers.Dense(8, input_dim=3, kernel_regularizer="l1_l2", bias_regularizer=layers.l1(0.2)))
    m.add(layers.Dense(1, activation="sigmoid", kernel_regularizer="L2"))
    assert m._factors() == ([0.01, 0.0, 0.01, 0.0], [0.01, 0.2, 0.0, 0.0])
    assert m._l2() == [0.01, 0.0, 0.01, 0.0]
    fac = StackedRecurrentFactory(4, 1, num_layers=1, num_units=8,
                                  layer_kws=dict(kernel_regularizer="l1", recurrent_regularizer=layers.L1L2(0.5, 0.25)))
    l2, l1 = fac._factors()
    assert l2 == [0.0, 0.25, 0.0, 0.0, 0.0] and l1 == [0.01, 0.5, 0.0, 0.0, 0.0]


def test_header_has_the_prototypes():
    with open(os.path.join(ROOT, "include", "bore_b200.h")) as fh:
        text = fh.read()
    assert re.search(r"int bore_mlp_set_l1_regularizers\(bore_mlp \*h, const float \*l1_kernel_host, "
                     r"const float \*l1_bias_host\);", text)
    assert re.search(r"int bore_lstm_set_l1_regularizers\(bore_lstm \*h, const float \*l1_per_array_host\);", text)
    assert int(re.search(r"#define BORE_ABI_VERSION (\d+)", text).group(1)) == 1
