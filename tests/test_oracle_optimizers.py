"""The Keras optimizers RMSprop, Adagrad, Adadelta, Adamax and Nadam: the oracle's rules (tests/optimizer_oracle.py)
against an independent torch-CPU implementation in fp64 -- ``torch.optim`` where its update is the same rule in
exact arithmetic, a hand-written update where torch differs -- and the host-side surface (class names, defaults,
refusals, the C enum and the native argument checks).  CPU only."""
import ctypes as C
import os
import re

import numpy as np
import pytest
import torch

from oracle import keras_lstm as kl, keras_mlp as km
import optimizer_oracle as oo
from bore_b200 import layers

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

# every kind, and the configurations that take another branch of its rule or non-default hyper-parameters
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
    "adam_custom": dict(learning_rate=3e-3, beta_1=0.8, beta_2=0.99, epsilon=1e-6),
}


def make(name):
    return type(layers.optimizer_spec(name.split("_")[0]))(**CONFIGS[name])


class _Hand(torch.optim.Optimizer):
    """The rules torch.optim states differently: RMSprop with momentum (eps inside the root), Adamax (torch puts
    eps inside the max) and Keras' Adam (eps outside the bias correction)."""

    def __init__(self, params, spec):
        super().__init__(params, {})
        self.spec, self.t = spec, 0

    @torch.no_grad()
    def step(self):
        o, self.t = self.spec, self.t + 1
        for p in self.param_groups[0]["params"]:
            g, st = p.grad, self.state[p]
            if not st:
                st["a"], st["b"] = torch.zeros_like(p), torch.zeros_like(p)
            a, b = st["a"], st["b"]
            if o.kind == "rmsprop":
                a.mul_(o.rho).add_((1 - o.rho) * g * g)
                b.mul_(o.momentum).add_(o.learning_rate * g / torch.sqrt(a + o.epsilon))
                p.sub_(b)
            elif o.kind == "adamax":
                a.mul_(o.beta_1).add_((1 - o.beta_1) * g)
                torch.maximum(o.beta_2 * b, g.abs(), out=b)
                p.sub_(o.learning_rate / (1 - o.beta_1 ** self.t) * a / (b + o.epsilon))
            else:
                a.mul_(o.beta_1).add_((1 - o.beta_1) * g)
                b.mul_(o.beta_2).add_((1 - o.beta_2) * g * g)
                lr_t = o.learning_rate * np.sqrt(1 - o.beta_2 ** self.t) / (1 - o.beta_1 ** self.t)
                p.sub_(lr_t * a / (torch.sqrt(b) + o.epsilon))


def torch_optimizer(params, o):
    """torch.optim's own optimizer where it runs the same rule in exact arithmetic (checked against torch's
    documented algorithms: RMSprop's square_avg / grad_avg, Adagrad's state_sum started at
    initial_accumulator_value with lr_decay 0, Adadelta's acc_delta, NAdam's mu_product with momentum_decay
    4e-3), else the hand-written rule."""
    if o.kind == "rmsprop" and o.momentum == 0:
        return torch.optim.RMSprop(params, lr=o.learning_rate, alpha=o.rho, eps=o.epsilon, centered=o.centered)
    if o.kind == "adagrad":
        return torch.optim.Adagrad(params, lr=o.learning_rate, initial_accumulator_value=o.initial_accumulator_value,
                                   eps=o.epsilon)
    if o.kind == "adadelta":
        return torch.optim.Adadelta(params, lr=o.learning_rate, rho=o.rho, eps=o.epsilon)
    if o.kind == "nadam":
        return torch.optim.NAdam(params, lr=o.learning_rate, betas=(o.beta_1, o.beta_2), eps=o.epsilon,
                                 momentum_decay=4e-3)
    return _Hand(params, o)


def _torch_mlp(ws, acts, X):
    h = X
    for l, a in enumerate(acts):
        h = h @ ws[2 * l] + ws[2 * l + 1]
        if l < len(acts) - 1:
            h = {"elu": torch.nn.functional.elu, "tanh": torch.tanh, "relu": torch.relu}[a](h)
    return h


def _torch_lstm(ws, X):
    """Stacked tanh LSTM (gates i, f, c, o) + Dense, no mask: logits (B, T)."""
    L, U = (len(ws) - 2) // 3, ws[1].shape[0]
    seq = X
    for l in range(L):
        K, R, b = ws[3 * l: 3 * l + 3]
        h = torch.zeros(X.shape[0], U, dtype=X.dtype)
        c = torch.zeros_like(h)
        outs = []
        for t in range(X.shape[1]):
            zz = seq[:, t] @ K + h @ R + b
            i, f, o = torch.sigmoid(zz[:, :U]), torch.sigmoid(zz[:, U:2 * U]), torch.sigmoid(zz[:, 3 * U:])
            c = f * c + i * torch.tanh(zz[:, 2 * U:3 * U])
            h = o * torch.tanh(c)
            outs.append(h)
        seq = torch.stack(outs, dim=1)
    return (seq @ ws[-2] + ws[-1])[..., 0]


def _torch_fit(w0, loss_fn, N, epochs, batch, perms, o, l2):
    ws = [torch.tensor(a, requires_grad=True) for a in w0]
    opt = torch_optimizer(ws, o)
    hist = []
    for e in range(epochs):
        tot = 0.0
        for s in range(0, N, batch):
            idx = torch.as_tensor(perms[e][s:s + batch])
            loss = loss_fn(ws, idx) + sum(l2 * (a * a).sum() for a in ws)
            opt.zero_grad()
            loss.backward()
            opt.step()
            tot += float(loss.detach()) * len(idx)
        hist.append(tot / N)
    return np.array(hist), [a.detach().numpy() for a in ws]


@pytest.mark.parametrize("name", sorted(CONFIGS))
@pytest.mark.parametrize("dims,acts,l2", [([4, 16, 8, 1], ["elu", "tanh", "sigmoid"], 0.0),
                                          ([3, 12, 1], ["relu", "linear"], 1e-3)])
def test_mlp_fit_vs_torch(name, dims, acts, l2):
    """100 steps (25 epochs x 4 batches) of the oracle fit loop under the kind's rule."""
    o = make(name)
    rs = np.random.RandomState(3)
    N, E, B = 100, 25, 25
    X = rs.uniform(-1.5, 1.5, size=(N, dims[0]))
    y = np.sum((X - 0.3) ** 2, axis=1)
    z = (y < np.quantile(y, 0.3)).astype(np.float64)
    perms = np.stack([rs.permutation(N) for _ in range(E)])
    w0 = km.init_weights(dims, 5, np.float64)
    w = [a.copy() for a in w0]
    with oo.installed():
        hist, st = km.fit(w, acts, X, z, E, B, perms, adam=oo.state_for(w, o, np.float64), l2=l2,
                          dtype=np.float64)
    assert st.t == 100
    Xt, zt = torch.tensor(X), torch.tensor(z).reshape(-1, 1)
    bce = torch.nn.functional.binary_cross_entropy_with_logits
    hist_t, wt = _torch_fit(w0, lambda ws, idx: bce(_torch_mlp(ws, acts, Xt[idx]), zt[idx]), N, E, B, perms, o, l2)
    assert np.abs(hist - hist_t).max() <= 1e-10
    assert max(np.abs(a - b).max() for a, b in zip(w, wt)) <= 1e-10
    assert max(np.abs(a - b).max() for a, b in zip(w, w0)) > 1e-4  # the rule moved the weights


@pytest.mark.parametrize("name", sorted(CONFIGS))
def test_lstm_fit_vs_torch(name):
    """100 steps (50 epochs x 2 batches) of keras_lstm's fit loop under the kind's rule."""
    o = make(name)
    D, U, L, T, N, E, B = 4, 8, 2, 3, 40, 50, 20
    rs = np.random.RandomState(7)
    X = rs.uniform(size=(N, T, D))
    Y = (rs.uniform(size=(N, T, 1)) < 0.4).astype(np.float64)
    perms = np.stack([rs.permutation(N) for _ in range(E)])
    w0 = kl.init_weights(D, U, L, seed=8, dtype=np.float64)
    w = [a.copy() for a in w0]
    with oo.installed():
        hist, st = kl.fit(w, "tanh", X, Y, E, B, perms, mask_value=-1e9, adam=oo.state_for(w, o, np.float64),
                          dtype=np.float64)
    assert st.t == 100
    Xt, Yt = torch.tensor(X), torch.tensor(Y[..., 0])
    bce = torch.nn.functional.binary_cross_entropy_with_logits
    hist_t, wt = _torch_fit(w0, lambda ws, idx: bce(_torch_lstm(ws, Xt[idx]), Yt[idx]), N, E, B, perms, o, 0.0)
    assert np.abs(hist - hist_t).max() <= 1e-10
    assert max(np.abs(a - b).max() for a, b in zip(w, wt)) <= 1e-10


def test_installed_keeps_adam():
    """Adam states still reach the oracle's own function, and the name is restored on exit."""
    w = km.init_weights([3, 4, 1], 0, np.float64)
    g = [np.ones_like(a) for a in w]
    w1, w2 = [a.copy() for a in w], [a.copy() for a in w]
    s1, s2 = km.AdamState(w1), km.AdamState(w2)
    km.adam_apply(w1, g, s1, np.float64)
    with oo.installed():
        km.adam_apply(w2, g, s2, np.float64)
    assert km.adam_apply is oo._KM_ADAM
    assert all(np.array_equal(a, b) for a, b in zip(w1, w2))


def test_padding_stays_zero():
    """A parameter with a zero gradient and zero slots stays exactly zero under every rule (the kernels' padding),
    in fp32 as the kernels compute."""
    for name in CONFIGS:
        o = make(name)
        w = [np.zeros(3, np.float32)]
        st = oo.state_for(w, o, np.float32)
        if isinstance(st, km.AdamState):
            continue
        st.s0 = [np.zeros(3, np.float32)]  # padding: zero slots whatever the initial value of real ones
        with oo.installed():
            for _ in range(5):
                km.adam_apply(w, [np.zeros(3, np.float32)], st, np.float32)
        assert np.array_equal(w[0], np.zeros(3, np.float32)) and np.isfinite(st.s1[0]).all(), name


def test_names_defaults_and_refusals():
    spec = layers.optimizer_spec
    # names are case-insensitive, as keras.optimizers.get takes them; the Keras 2.5 defaults
    assert isinstance(spec("RMSprop"), layers.RMSprop) and isinstance(spec("NADAM"), layers.Nadam)
    r = spec("rmsprop")
    assert (r.learning_rate, r.rho, r.momentum, r.epsilon, r.centered) == (1e-3, 0.9, 0.0, 1e-7, False)
    a = spec("adagrad")
    assert (a.learning_rate, a.initial_accumulator_value, a.epsilon) == (1e-3, 0.1, 1e-7)
    d = spec("adadelta")
    assert (d.learning_rate, d.rho, d.epsilon) == (1e-3, 0.95, 1e-7)
    for cls in (layers.Adam, layers.Adamax, layers.Nadam):
        o = cls()
        assert (o.learning_rate, o.beta_1, o.beta_2, o.epsilon) == (1e-3, 0.9, 0.999, 1e-7)
    assert layers.Adam(amsgrad=False).amsgrad is False
    inst = layers.Adamax(learning_rate=0.01)
    assert spec(inst) is inst
    # the C hyper-parameter arrays
    assert layers.RMSprop(centered=True).hyper() == (1, [1e-3, 0.9, 0.0, 1e-7, 0.0, 0.0, 1.0])
    assert layers.Adagrad().hyper() == (2, [1e-3, 0.0, 0.0, 1e-7, 0.0, 0.1, 0.0])
    assert layers.Nadam(beta_2=0.99).hyper() == (5, [1e-3, 0.9, 0.99, 1e-7, 0.0, 0.0, 0.0])
    # refused, each with its reason
    with pytest.raises(NotImplementedError, match="no training kernel"):
        spec("sgd")
    with pytest.raises(NotImplementedError, match="Ftrl"):
        spec("Ftrl")
    with pytest.raises(ValueError, match="nadam"):
        spec("lamb")
    with pytest.raises(NotImplementedError, match="third slot"):
        layers.Adam(amsgrad=True)
    with pytest.raises(NotImplementedError, match="third slot"):
        layers.RMSprop(centered=True, momentum=0.5)
    for kw in ("decay", "clipnorm", "clipvalue", "global_clipnorm"):
        with pytest.raises(TypeError, match=kw):
            layers.Nadam(**{kw: 0.1})
    with pytest.raises(NotImplementedError, match="schedule"):
        layers.RMSprop(learning_rate=lambda step: 1e-3)


def test_sgd_still_refused_on_both_surfaces():
    from bore_b200.layers import BinaryCrossentropy, Dense
    from bore_b200.models import MaximizableSequential, StackedRecurrentFactory
    r = MaximizableSequential()
    r.add(Dense(16, activation="relu")); r.add(Dense(1, activation="sigmoid"))
    for name in ("adagrad", "Nadam", layers.RMSprop(momentum=0.5)):
        r.compile(optimizer=name, loss="binary_crossentropy")
    with pytest.raises(NotImplementedError):
        r.compile(optimizer="sgd", loss="binary_crossentropy")
    net = StackedRecurrentFactory(4, 1, num_layers=2, num_units=8).build_many_to_many(mask_value=-1.0)
    net.compile(optimizer=layers.Adam(learning_rate=3e-3), loss=BinaryCrossentropy(from_logits=True))
    net.compile(optimizer="adadelta", loss=BinaryCrossentropy(from_logits=True))
    with pytest.raises(NotImplementedError):
        net.compile(optimizer="sgd", loss=BinaryCrossentropy(from_logits=True))


def test_plugin_constructors():
    """BORE and BOREHyperband refuse an optimizer the kernels do not run when they are built."""
    from bore_b200.plugins.hpbandster import BORE, BOREHyperband
    from bore_b200.plugins.hpbandster._compat import CS
    space = CS.ConfigurationSpace(seed=0)
    space.add_hyperparameter(CS.UniformFloatHyperparameter("x", lower=0.0, upper=1.0))
    assert BORE(space, optimizer="rmsprop").config_generator.optimizer == "rmsprop"
    assert BOREHyperband(space, optimizer="nadam").config_generator.optimizer == "nadam"
    for cls in (BORE, BOREHyperband):
        with pytest.raises(NotImplementedError, match="SGD"):
            cls(space, optimizer="sgd")
        with pytest.raises(ValueError):
            cls(space, optimizer="lamb")


def test_header_enum_matches_codes():
    with open(os.path.join(ROOT, "include", "bore_b200.h")) as fh:
        text = fh.read()
    enum = dict((k.lower(), int(v)) for k, v in re.findall(r"BORE_OPT_([A-Z]+) = (\d+)", text))
    assert enum == layers.OPT_CODES
    assert int(re.search(r"#define BORE_OPT_NHP (\d+)", text).group(1)) == len(layers.Adam().hyper()[1])


def test_native_argument_checks(native_lib):
    """bore_{mlp,lstm}_set_optimizer_kind check the kind and the ranges before the handle (no device needed)."""
    lib = native_lib

    def call(fn, kind, hp):
        arr = (C.c_float * 7)(*hp)
        rc = getattr(lib, fn)(None, kind, arr)
        return rc, lib.bore_last_error().decode()

    for fn in ("bore_mlp_set_optimizer_kind", "bore_lstm_set_optimizer_kind"):
        good = {k: layers.optimizer_spec(k).hyper() for k in layers.OPT_CODES}
        for k, (code, hp) in good.items():
            rc, msg = call(fn, code, hp)
            assert rc != 0 and msg == "NULL handle", (k, msg)  # every check passed
        for code in (-1, 6):
            rc, msg = call(fn, code, good["adam"][1])
            assert rc != 0 and f"unknown optimizer kind {code}" in msg
        bad = [(1, [1e-3, 0.9, 0, 1e-7, 0.5, 0, 1], "third slot"), (2, [1e-3, 0, 0, 0.0, 0, 0.1, 0], "epsilon"),
               (3, [1e-3, 1.0, 0, 1e-7, 0, 0, 0], "rho"), (4, [0.0, 0.9, 0.999, 1e-7, 0, 0, 0], "learning_rate"),
               (5, [1e-3, 0.9, 1.5, 1e-7, 0, 0, 0], "beta_2"), (2, [1e-3, 0, 0, 1e-7, 0, -1, 0], "initial_acc")]
        for code, hp, what in bad:
            rc, msg = call(fn, code, hp)
            assert rc != 0 and what in msg, (code, msg)
