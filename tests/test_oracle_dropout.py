"""Keras Dropout between Dense layers: the mask (Philox4x32-10 known answers, keep fraction, independence across layer,
model, step and seed), the oracle's rule (tests/dropout_oracle.py) against an independent torch-CPU autograd fit in
fp64 with the same masks as fixed tensors, and the host-side surface: the layer, its placement rules, Sequential's
bookkeeping, seed reproducibility and the native argument checks (no device needed)."""
import ctypes as C

import numpy as np
import pytest
import torch

from oracle import keras_mlp as km
import dropout_oracle as do
import optimizer_oracle as oo
from helpers import synthetic_targets
from bore_b200 import layers
from bore_b200.layers import Dense, Dropout


# ------------------------------------------------------------------------------------------------ the mask
@pytest.mark.parametrize("ctr,key,out", [
    ((0, 0, 0, 0), (0, 0), (0x6627e8d5, 0xe169c58d, 0xbc57ac4c, 0x9b00dbd8)),
    ((0xffffffff,) * 4, (0xffffffff,) * 2, (0x408f276d, 0x41c83b0e, 0xa20bc7c6, 0x6d5451fd)),
    ((0x243f6a88, 0x85a308d3, 0x13198a2e, 0x03707344), (0xa4093822, 0x299f31d0),
     (0xd16cfe09, 0x94fdcceb, 0x5001e420, 0x24126ea1)),
])
def test_philox_known_answers(ctr, key, out):
    assert tuple(int(v) for v in do.philox4x32_10(ctr, key)) == out


@pytest.mark.parametrize("rate", [0.1, 0.5])
def test_keep_fraction(rate):
    """10^6 draws (1000 samples x 1000 units of one step) keep 1 - rate of the units within a 6-sigma bound."""
    n = 10 ** 6
    kept = do.keep_mask(2, 12345, 1000, 1000, rate, 77, 3).sum()
    p = 1.0 - float(np.float32(rate))
    assert abs(kept - n * p) <= 6 * np.sqrt(n * p * (1 - p)), kept


def test_masks_differ():
    base = dict(l=1, t=7, nb=64, width=64, rate=0.5, seed=11, m=0)
    m0 = do.keep_mask(**base)
    for k, v in (("l", 2), ("m", 1), ("t", 8), ("t", 7 + 2 ** 32), ("seed", 12)):
        other = do.keep_mask(**dict(base, **{k: v}))
        assert 0.3 < np.mean(other != m0) < 0.7, k  # independent masks disagree on about half the units
    assert np.array_equal(do.keep_mask(**base), m0)


def test_mask_layout():
    """Units 4q .. 4q + 3 of a sample are the four words of one Philox call."""
    w = do.philox4x32_10((5, 0, 3, 65536 * 1 + 2), (9, 4))
    u = do.uniforms(1, 5, 3, np.arange(8, 12), 9, 4)
    assert np.array_equal(u, (w >> np.uint32(8)).astype(np.float64) * 2.0 ** -24)


# ------------------------------------------------------------------------------------------------ the rule
def _torch_fit(w0, acts, X, z, E, B, perms, rates, seeds, kind, l2):
    """fp64 torch autograd: h~ = act(h W + b) * scale * mask (masks fixed), the textbook Adam / RMSprop."""
    ws = [torch.tensor(a, dtype=torch.float64, requires_grad=True) for a in w0]
    s0 = [torch.zeros_like(w) for w in ws]
    s1 = [torch.zeros_like(w) for w in ws]
    f = {"elu": torch.nn.functional.elu, "tanh": torch.tanh, "sigmoid": lambda v: v, "linear": lambda v: v}
    Xt, zt = torch.tensor(X, dtype=torch.float64), torch.tensor(z, dtype=torch.float64)
    t = 0
    hist = []
    N = X.shape[0]
    for e in range(E):
        tot = 0.0
        for s in range(0, N, B):
            idx = perms[e][s:s + B]
            h = Xt[idx]
            for l in range(len(acts)):
                h = f[acts[l]](h @ ws[2 * l] + ws[2 * l + 1])
                if l < len(acts) - 1 and rates[l] > 0:
                    mask = torch.tensor(do.keep_mask(l, t, len(idx), h.shape[1], rates[l], seeds[l], 0))
                    h = h * float(do.scale_of(rates[l])) * mask
            loss = torch.nn.functional.binary_cross_entropy_with_logits(h[:, 0], zt[idx])
            loss = loss + sum(l2 * (w * w).sum() for w in ws)
            grads = torch.autograd.grad(loss, ws)
            tot += loss.item() * len(idx)
            t += 1
            with torch.no_grad():
                for i, (w, g) in enumerate(zip(ws, grads)):
                    if kind == "adam":
                        s0[i] = 0.9 * s0[i] + 0.1 * g
                        s1[i] = 0.999 * s1[i] + 0.001 * g * g
                        alpha = 1e-3 * np.sqrt(1 - 0.999 ** t) / (1 - 0.9 ** t)
                        w -= alpha * s0[i] / (torch.sqrt(s1[i]) + 1e-7)
                    else:
                        s0[i] = 0.9 * s0[i] + 0.1 * g * g
                        w -= 1e-3 * g / (torch.sqrt(s0[i]) + 1e-7)
        hist.append(tot / N)
    return np.array(hist), [w.detach().numpy() for w in ws]


@pytest.mark.parametrize("act,kind,l2", [("elu", "adam", 0.0), ("tanh", "rmsprop", 1e-3), ("elu", "rmsprop", 0.0),
                                         ("tanh", "adam", 1e-3)])
def test_oracle_against_torch(act, kind, l2):
    """100 fp64 steps (5 epochs x 20 batches) of a two-hidden-layer MLP, dropout 0.3 and 0.5."""
    dims, acts = [5, 16, 12, 1], [act, act, "linear"]
    rs = np.random.RandomState(3)
    N, B, E = 300, 15, 5
    X = rs.uniform(size=(N, 5))
    y = synthetic_targets(X)
    z = (y < np.quantile(y, 0.3)).astype(np.float64)
    perms = np.stack([rs.permutation(N) for _ in range(E)])
    rates, seeds = [0.3, 0.5], [123, 2 ** 32 - 1]
    w0 = km.init_weights(dims, 4, np.float64)
    h_t, w_t = _torch_fit(w0, acts, X, z, E, B, perms, rates, seeds, kind, l2)
    w = [a.copy() for a in w0]
    st = km.AdamState(w) if kind == "adam" else oo.RMSpropState(w)
    with oo.installed():
        h_o, st = do.fit(w, acts, X, z, E, B, perms, rates, seeds, state=st, l2=l2, dtype=np.float64)
    assert st.t == 100
    assert np.abs(h_o - h_t).max() <= 1e-10
    for a, b in zip(w, w_t):
        assert np.abs(a - b).max() <= 1e-10


def test_rate_zero_is_no_dropout():
    dims, acts = [4, 8, 8, 1], ["relu", "relu", "sigmoid"]
    rs = np.random.RandomState(1)
    X, z = rs.uniform(size=(50, 4)), (rs.uniform(size=50) < 0.4).astype(np.float32)
    perms = np.stack([rs.permutation(50) for _ in range(3)])
    w0 = km.init_weights(dims, 2)
    w1, w2 = [a.copy() for a in w0], [a.copy() for a in w0]
    h1, _ = do.fit(w1, acts, X, z, 3, 16, perms, [0.0, 0.0], [1, 2])
    h2, _ = km.fit(w2, acts, X, z, 3, 16, perms)
    assert np.array_equal(h1, h2) and all(np.array_equal(a, b) for a, b in zip(w1, w2))


# ------------------------------------------------------------------------------------------------ the layer
def test_layer():
    d = Dropout(0.25)
    assert (d.rate, d.noise_shape, d.seed) == (0.25, None, None)
    assert Dropout(0.0, seed=2 ** 32 - 1).seed == 2 ** 32 - 1
    assert Dropout(rate=0.5, noise_shape=None, seed=3).seed == 3
    for bad in (1.0, 1.5, -0.1, float("nan"), float("inf")):
        with pytest.raises(ValueError, match="rate"):
            Dropout(bad)
    for bad in (-1, 2 ** 32, 1.5):
        with pytest.raises(ValueError, match="seed"):
            Dropout(0.1, seed=bad)
    with pytest.raises(NotImplementedError, match="noise_shape"):
        Dropout(0.1, noise_shape=(None, 1))
    with pytest.raises(TypeError):
        Dropout(0.1, training=True)
    import bore_b200
    assert bore_b200.Dropout is Dropout


def test_placement():
    from bore_b200.models import Sequential
    m = Sequential()
    with pytest.raises(NotImplementedError, match="input dropout"):
        m.add(Dropout(0.2))
    m.add(Dense(8, activation="relu", input_dim=3))
    m.add(Dropout(0.2))
    with pytest.raises(NotImplementedError, match="in a row"):
        m.add(Dropout(0.2))
    m.add(Dense(1, activation="sigmoid"))
    m.add(Dropout(0.1))  # add cannot know that the Dense before it was the output layer
    with pytest.raises(NotImplementedError, match="must be followed by a Dense layer"):
        m.compile(optimizer="adam", loss="binary_crossentropy")
    with pytest.raises(NotImplementedError, match="must be followed by a Dense layer"):
        m._engine()
    with pytest.raises(NotImplementedError, match="Dense and Dropout"):
        m.add("conv")
    for ls, what in (([Dropout(0.1), Dense(1, input_dim=2)], "input dropout"),
                     ([Dense(4, input_dim=2), Dropout(0.1), Dropout(0.1), Dense(1)], "in a row"),
                     ([Dense(4, input_dim=2), Dense(1), Dropout(0.1)], "must be followed by a Dense layer")):
        with pytest.raises(NotImplementedError, match=what):
            layers.split_dropout(ls)


def test_sequential_bookkeeping():
    from bore_b200.models import Sequential
    m = Sequential([Dense(8, activation="elu", input_dim=3, kernel_regularizer="l2"), Dropout(0.2),
                    Dense(6, activation="elu", bias_regularizer="l1"), Dropout(0.0), Dense(1, activation="sigmoid")])
    plain = Sequential([Dense(8, activation="elu", input_dim=3, kernel_regularizer="l2"),
                        Dense(6, activation="elu", bias_regularizer="l1"), Dense(1, activation="sigmoid")])
    assert len(m.layers) == 5 and m.input_dim == 3
    assert m.count_params() == plain.count_params() == 3 * 8 + 8 + 8 * 6 + 6 + 6 + 1
    assert m._factors() == plain._factors()
    dense, after = m._split()
    assert [d.units for d in dense] == [8, 6, 1] and [a.rate for a in after] == [0.2, 0.0]
    lines = []
    m.summary(print_fn=lines.append)
    assert any(ln.startswith("dropout_0 (Dropout)") and "output=(None, 8)" in ln and "params=0" in ln for ln in lines)
    assert any(ln.startswith("dropout_1 (Dropout)") and "output=(None, 6)" in ln for ln in lines)
    assert sum(ln.startswith("dense_") for ln in lines) == 3
    assert lines[-1] == f"Total params: {plain.count_params()}"
    m.compile(optimizer="adam", loss="binary_crossentropy")  # the final activation is the last Dense layer's


class _FakeNet:
    """Stands in for NativeMLP: records what the surface sends."""

    def __init__(self, dims, acts, n_models=1, device=None):
        self.dims, self.acts, self.D, self.calls = dims, acts, dims[0], []

    def set_weights(self, ws, model=0):
        self.calls.append(("weights", [np.array(w) for w in ws]))

    def set_dropout(self, rates, seeds):
        self.calls.append(("dropout", list(rates), list(seeds)))

    def set_optimizer_kind(self, optimizer):
        self.calls.append(("optimizer",))

    def set_regularizers(self, l2, l1=None):
        self.calls.append(("regularizers",))


def _sequential(seed, rates, seeds=(None, None)):
    from bore_b200.models import Sequential
    m = Sequential(seed=seed)
    m.add(Dense(8, activation="relu", input_dim=3))
    m.add(Dropout(rates[0], seed=seeds[0]))
    m.add(Dense(8, activation="relu"))
    m.add(Dropout(rates[1], seed=seeds[1]))
    m.add(Dense(1, activation="sigmoid"))
    return m


def test_seeds(monkeypatch):
    """seed=None draws from the model's RandomState once, after the initial weights, in layer order; rate-0 layers
    draw nothing and send nothing; an explicit seed is sent as given."""
    from bore_b200 import engine
    monkeypatch.setattr(engine, "NativeMLP", _FakeNet)
    a, b = _sequential(7, (0.2, 0.3))._engine(), _sequential(7, (0.2, 0.3))._engine()
    assert [c[0] for c in a.calls] == ["weights", "dropout"]
    assert a.calls[1] == b.calls[1]
    rs = np.random.RandomState(7)
    for fi, fo in ((3, 8), (8, 8), (8, 1)):
        rs.uniform(size=(fi, fo))
    s0, s1 = (int(rs.randint(0, 2 ** 32, dtype=np.int64)) for _ in range(2))
    assert a.calls[1] == ("dropout", [0.2, 0.3], [s0, s1])
    assert all(np.array_equal(x, y) for x, y in zip(a.calls[0][1], _sequential(7, (0.0, 0.0))._engine().calls[0][1]))
    c = _sequential(7, (0.0, 0.3), seeds=(None, 5))._engine()
    assert c.calls[1] == ("dropout", [0.0, 0.3], [0, 5])
    d = _sequential(7, (0.0, 0.3))._engine()
    assert d.calls[1] == ("dropout", [0.0, 0.3], [0, s0])  # the rate-0 layer drew nothing
    assert [x[0] for x in _sequential(7, (0.0, 0.0))._engine().calls] == ["weights"]  # Dropout(0.0): nothing sent
    assert _sequential(8, (0.2, 0.3))._engine().calls[1] != a.calls[1]


def test_batched_surface_checks(monkeypatch):
    from bore_b200 import batched
    monkeypatch.setattr(batched, "NativeMLP", _FakeNet)
    m = batched.BatchedMaximizableSequential([Dense(8, activation="relu", input_dim=3), Dropout(0.4, seed=9),
                                              Dense(1, activation="sigmoid")], n_problems=3, seed=1)
    assert m.dims == [3, 8, 1] and m._net.calls[-1] == ("dropout", [0.4], [9])
    assert [c[0] for c in m._net.calls] == ["weights"] * 3 + ["dropout"]
    for ls, what in (([Dropout(0.1), Dense(1, input_dim=2)], "input dropout"),
                     ([Dense(4, input_dim=2), Dropout(0.1), Dropout(0.1), Dense(1)], "in a row"),
                     ([Dense(4, input_dim=2), Dense(1), Dropout(0.1)], "must be followed by a Dense layer")):
        with pytest.raises(NotImplementedError, match=what):
            batched.BatchedMaximizableSequential(ls, n_problems=2)


# ------------------------------------------------------------------------------------------------ the C ABI
def test_native_argument_checks(native_lib):
    """bore_mlp_set_dropout checks its arguments before the handle (no device needed)."""
    lib = native_lib

    def call(n, rates, seeds=None, null=False):
        r = (C.c_float * max(1, len(rates)))(*rates)
        s = (C.c_uint32 * max(1, n))(*(seeds or [1] * n))
        rc = lib.bore_mlp_set_dropout(None, n, None if null else r, None if null else s)
        return rc, lib.bore_last_error().decode()

    for n, rates in ((0, []), (1, [0.0]), (2, [0.5, 0.999]), (7, [0.1] * 7)):
        rc, msg = call(n, rates)
        assert rc != 0 and msg == "NULL handle", (n, rates, msg)  # every check passed
    assert call(0, [], null=True) == (call(0, [], null=True)[0], "NULL handle")
    for n, rates, what in ((-1, [], "outside [0, 7]"), (8, [0.1] * 8, "outside [0, 7]"), (1, [1.0], "in [0, 1)"),
                           (1, [-0.1], "in [0, 1)"), (2, [0.1, float("nan")], "hidden layer 1"),
                           (1, [float("inf")], "in [0, 1)")):
        rc, msg = call(n, rates)
        assert rc != 0 and what in msg, (n, rates, msg)
    rc, msg = call(1, [0.1], null=True)
    assert rc != 0 and "NULL argument" in msg
