"""The activations selu, softplus, softsign, hard_sigmoid and exponential: the oracle's rules
(tests/activation_oracle.py) against an independent torch-CPU autograd implementation written from the TF
2.5 formulas in fp64, the fp32 deviation of the kernels' through-output derivative from TF's own rule, and
the host-side surface (layer names, the C enum, the create-time range checks).  CPU only."""
import ctypes as C
import os
import re

import numpy as np
import pytest
import torch

from oracle import keras_lstm as kl, keras_mlp as km
import activation_oracle as ao

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(autouse=True, scope="module")
def _extended_oracle():
    with ao.installed():
        yield


def _t_act(name, a):
    """fp64 torch forms of the TF 2.5 ops (not F.hardsigmoid: that is relu6(x + 3) / 6; not F.softplus:
    its own threshold of 20)."""
    if name == "linear":
        return a
    if name == "relu":
        return torch.relu(a)
    if name == "elu":
        return torch.where(a > 0, a, torch.expm1(torch.clamp(a, max=0.0)))
    if name == "sigmoid":
        return torch.sigmoid(a)
    if name == "tanh":
        return torch.tanh(a)
    if name == "selu":
        return torch.where(a > 0, ao.SELU_SCALE * a, ao.SELU_SCALE_ALPHA * torch.expm1(torch.clamp(a, max=0.0)))
    if name == "softplus":
        thr = float(ao.softplus_threshold(np.float64))
        return torch.where(a > -thr, a, torch.where(a < thr, torch.exp(a), torch.log(torch.exp(torch.clamp(a, max=-thr)) + 1)))
    if name == "softsign":
        return a / (torch.abs(a) + 1)
    if name == "hard_sigmoid":
        return torch.clamp(0.2 * a + 0.5, 0.0, 1.0)
    if name == "exponential":
        return torch.exp(a)
    raise ValueError(name)


# hidden activations of the test nets: each new one alone, and one net that mixes them
NETS = {a: ([4, 12, 10, 1], [a, a, "sigmoid"]) for a in ao.NEW}
NETS["mixed"] = ([5, 16, 12, 8, 1], ["selu", "softsign", "hard_sigmoid", "linear"])
NETS["mixed_exp"] = ([3, 8, 8, 1], ["softplus", "exponential", "sigmoid"])


def _torch_forward(ws, acts, X, last_linear=False):
    h = X
    for l, a in enumerate(acts):
        h = h @ ws[2 * l] + ws[2 * l + 1]
        if not (last_linear and l == len(acts) - 1):
            h = _t_act(a, h)
    return h


def _problem(dims, seed, N=90):
    rs = np.random.RandomState(seed)
    X = rs.uniform(-1.5, 1.5, size=(N, dims[0]))
    y = np.sum((X - 0.3) ** 2, axis=1)
    return X, y < np.quantile(y, 0.3), rs


@pytest.mark.parametrize("name", sorted(NETS))
@pytest.mark.parametrize("transform", ["identity", "sigmoid"])
def test_value_and_input_grad_vs_torch(name, transform):
    dims, acts = NETS[name]
    w = km.init_weights(dims, 1, np.float64)
    w = [a + 0.1 * np.random.RandomState(2).normal(size=a.shape) for a in w]  # non-zero biases
    X, _, _ = _problem(dims, 3)
    f, g = km.value_and_input_grad(w, acts, X, transform, True, np.float64)
    Xt = torch.tensor(X, requires_grad=True)
    u = _torch_forward([torch.tensor(a) for a in w], acts, Xt)[:, 0]
    ft = {"identity": lambda t: t, "sigmoid": torch.sigmoid}[transform](-u)
    ft.sum().backward()
    assert np.allclose(f, ft.detach().numpy(), rtol=1e-12, atol=1e-14)
    assert np.abs(g - Xt.grad.numpy()).max() <= 1e-10 * max(1.0, np.abs(g).max())


@pytest.mark.parametrize("name", sorted(NETS))
@pytest.mark.parametrize("l2", [0.0, 1e-3])
def test_weight_grads_and_fit_vs_torch(name, l2):
    dims, acts = NETS[name]
    fit_acts = list(acts[:-1]) + ["sigmoid" if acts[-1] == "sigmoid" else "linear"]
    X, z, rs = _problem(dims, 4)
    w0 = km.init_weights(dims, 5, np.float64)
    loss, grads = km.loss_and_weight_grads(w0, fit_acts, X, z, l2, np.float64)
    wt = [torch.tensor(a, requires_grad=True) for a in w0]
    u = _torch_forward(wt, fit_acts, torch.tensor(X), last_linear=True)
    lt = torch.nn.functional.binary_cross_entropy_with_logits(u, torch.tensor(z, dtype=torch.float64).reshape(-1, 1))
    lt = lt + sum(l2 * (a * a).sum() for a in wt)
    gt = torch.autograd.grad(lt, wt)
    assert abs(float(loss) - lt.item()) <= 1e-12
    for a, b in zip(grads, gt):
        assert np.abs(a - b.numpy()).max() <= 1e-10 * max(1.0, np.abs(b.numpy()).max())
    # 100 Adam steps: 50 epochs of two batches (64 + 26)
    E, B = 50, 64
    perms = np.stack([rs.permutation(len(X)) for _ in range(E)])
    w = [a.copy() for a in w0]
    hist, adam = km.fit(w, fit_acts, X, z, E, B, perms, l2=l2, dtype=np.float64)
    hist_t, w_t = _torch_fit(w0, fit_acts, X, z, E, B, perms, l2)
    assert adam.t == 100
    assert np.abs(hist - hist_t).max() <= 1e-10
    assert max(np.abs(a - b).max() for a, b in zip(w, w_t)) <= 1e-10


def _torch_fit(w0, acts, X, z, epochs, batch, perms, l2, lr=1e-3, b1=0.9, b2=0.999, eps=1e-7):
    """Autograd gradients, torch's BCE-with-logits, textbook Adam (eps outside the bias correction)."""
    ws = [torch.tensor(a, requires_grad=True) for a in w0]
    m = [torch.zeros_like(a) for a in ws]
    v = [torch.zeros_like(a) for a in ws]
    Xt, zt = torch.tensor(X), torch.tensor(z, dtype=torch.float64).reshape(-1, 1)
    t, hist = 0, []
    for e in range(epochs):
        tot = 0.0
        perm = torch.as_tensor(perms[e])
        for s in range(0, len(X), batch):
            idx = perm[s:s + batch]
            u = _torch_forward(ws, acts, Xt[idx], last_linear=True)
            loss = torch.nn.functional.binary_cross_entropy_with_logits(u, zt[idx])
            loss = loss + sum(l2 * (a * a).sum() for a in ws)
            grads = torch.autograd.grad(loss, ws)
            tot += float(loss) * len(idx)
            t += 1
            lr_t = lr * np.sqrt(1.0 - b2 ** t) / (1.0 - b1 ** t)
            with torch.no_grad():
                for i, g in enumerate(grads):
                    m[i] = b1 * m[i] + (1.0 - b1) * g
                    v[i] = b2 * v[i] + (1.0 - b2) * g * g
                    ws[i] -= lr_t * m[i] / (torch.sqrt(v[i]) + eps)
        hist.append(tot / len(X))
    return np.array(hist), [a.detach().numpy() for a in ws]


def _torch_lstm(ws, activation, X):
    """Stacked LSTM (gates i, f, c, o) + Dense, no mask: logits (B, T)."""
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
            c = f * c + i * _t_act(activation, zz[:, 2 * U:3 * U])
            h = o * _t_act(activation, c)
            outs.append(h)
        seq = torch.stack(outs, dim=1)
    return (seq @ ws[-2] + ws[-1])[..., 0]


@pytest.mark.parametrize("activation", ["softplus", "selu"])
def test_lstm_vs_torch(activation):
    D, U, L, T, N = 4, 8, 2, 3, 40
    rs = np.random.RandomState(7)
    X = rs.uniform(size=(N, T, D))
    Y = (rs.uniform(size=(N, T, 1)) < 0.4).astype(np.float64)
    mask = np.ones((N, T), bool)
    w0 = kl.init_weights(D, U, L, seed=8, dtype=np.float64)
    # value and input gradient of the one-to-one network
    Xq = rs.uniform(size=(15, D))
    f, g = kl.value_and_input_grad(w0, activation, Xq, T, "sigmoid", True, np.float64)
    Xqt = torch.tensor(Xq, requires_grad=True)
    ft = torch.sigmoid(-_torch_lstm([torch.tensor(a) for a in w0], activation, Xqt[:, None, :].repeat(1, T, 1))[:, -1])
    ft.sum().backward()
    assert np.allclose(f, ft.detach().numpy(), rtol=1e-12, atol=1e-14)
    assert np.abs(g - Xqt.grad.numpy()).max() <= 1e-10 * max(1.0, np.abs(g).max())
    # weight gradients of the sequence loss
    loss, grads = kl.loss_and_weight_grads(w0, activation, X, Y, mask, None, np.float64)
    wt = [torch.tensor(a, requires_grad=True) for a in w0]
    lt = torch.nn.functional.binary_cross_entropy_with_logits(_torch_lstm(wt, activation, torch.tensor(X)),
                                                             torch.tensor(Y[..., 0]))
    for a, b in zip(grads, torch.autograd.grad(lt, wt)):
        assert np.abs(a - b.numpy()).max() <= 1e-10 * max(1.0, np.abs(b.numpy()).max())
    assert abs(float(loss) - float(lt)) <= 1e-12
    # 100 Adam steps (50 epochs x 2 batches)
    E, B = 50, 32
    perms = np.stack([rs.permutation(N) for _ in range(E)])
    w = [a.copy() for a in w0]
    hist, _ = kl.fit(w, activation, X, Y, E, B, perms, mask_value=-1e9, dtype=np.float64)
    ws = [torch.tensor(a, requires_grad=True) for a in w0]
    m = [torch.zeros_like(a) for a in ws]
    v = [torch.zeros_like(a) for a in ws]
    t, hist_t = 0, []
    for e in range(E):
        tot = 0.0
        for s in range(0, N, B):
            idx = torch.as_tensor(perms[e][s:s + B])
            lb = torch.nn.functional.binary_cross_entropy_with_logits(
                _torch_lstm(ws, activation, torch.tensor(X)[idx]), torch.tensor(Y[..., 0])[idx])
            gs = torch.autograd.grad(lb, ws)
            tot += float(lb) * len(idx)
            t += 1
            lr_t = 1e-3 * np.sqrt(1.0 - 0.999 ** t) / (1.0 - 0.9 ** t)
            with torch.no_grad():
                for i, gg in enumerate(gs):
                    m[i] = 0.9 * m[i] + 0.1 * gg
                    v[i] = 0.999 * v[i] + 0.001 * gg * gg
                    ws[i] -= lr_t * m[i] / (torch.sqrt(v[i]) + 1e-7)
        hist_t.append(tot / N)
    assert np.abs(hist - np.array(hist_t)).max() <= 1e-10
    assert max(np.abs(a - b.detach().numpy()).max() for a, b in zip(w, ws)) <= 1e-10


def _deviation_grid():
    """fp32 pre-activations: a dense sweep of [-1e3, 1e3] plus the softplus thresholds (+-13.942385) and the
    hard_sigmoid edges (+-2.5), each with its fp32 neighbours."""
    f = np.float32
    thr = ao.softplus_threshold(np.float32)
    pts = [np.linspace(-20, 20, 40001, dtype=f), np.geomspace(f(20), f(1e3), 2000).astype(f)]
    pts.append(-pts[-1])
    for c in (thr, -thr, f(2.5), f(-2.5)):
        pts.append(np.array([np.nextafter(c, f(-np.inf)), c, np.nextafter(c, f(np.inf))], f))
    return np.unique(np.concatenate(pts))


@pytest.mark.parametrize("name", ["softplus", "softsign", "hard_sigmoid", "selu", "exponential"])
def test_through_output_derivative_deviation(name):
    """The kernels' d act / d a from the fp32 output h, against the exact derivative at the fp32
    pre-activation (fp64): softplus and softsign differ by rounding, softsign's 1 - |h| cancelling for
    large |a|; hard_sigmoid only at the edges; selu and exponential are TF's own output-based rules."""
    a32 = _deviation_grid()
    h32 = ao.act(name, a32)
    d32 = ao.act_grad_from_output(name, h32).astype(np.float64)
    a64 = a32.astype(np.float64)
    if name == "softplus":
        with np.errstate(over="ignore"):
            exact = 1.0 / (1.0 + np.exp(-a64))
    elif name == "softsign":
        exact = 1.0 / (1.0 + np.abs(a64)) ** 2
    elif name == "hard_sigmoid":
        exact = ao.act_grad_from_features(name, a32).astype(np.float64)
    elif name == "selu":
        exact = np.where(a64 < 0, ao.SELU_SCALE_ALPHA * np.exp(a64), ao.SELU_SCALE)
    else:
        exact = np.exp(a64)
    with np.errstate(invalid="ignore"):
        err = np.abs(d32 - exact)
        rel = np.where(np.isfinite(exact) & (exact > 0), err / exact, 0.0)
    finite = np.isfinite(exact)
    if name == "hard_sigmoid":
        # differs from TF's closed interval only where 0.2 a + 0.5 rounds to exactly 0 or 1
        x = a32 * np.float32(0.2) + np.float32(0.5)
        assert np.array_equal(err > 0, (x == 0) | (x == 1))
        assert err.max() == pytest.approx(0.2)
    elif name == "softplus":
        # absolute deviation below 2^-23 everywhere; relative up to 7 % just above the lower threshold, where
        # TF's own fp32 log(exp(a) + 1) has already rounded h that much
        assert err[finite].max() < 1.2e-7, err[finite].max()
        assert rel[finite & (np.abs(a64) <= 5)].max() < 1e-5
    elif name == "softsign":
        # absolute deviation below 2^-23; the RELATIVE one grows with |a| as 1 - |h| cancels (9e-5 at 1e3)
        assert err.max() < 1.2e-7, err.max()
        assert rel[np.abs(a64) <= 10].max() < 2e-6
        assert 1e-5 < rel.max() < 2e-4
    elif name == "selu":
        # TF's SeluGrad formula itself; h + scale_alpha cancels for a << 0 (absolute deviation only)
        assert err[finite].max() < 2e-7, err[finite].max()
    else:
        ok = np.abs(a64) <= 80  # inside the fp32 range of exp, no denormals
        assert (rel[ok] < 1e-6).all()
    assert (d32 >= 0).all()


def test_layer_names():
    from bore_b200.layers import Dense, _ACTIVATIONS
    from bore_b200.recurrent import LSTMCell
    from bore_b200.models import DenseSequential
    from bore_b200.engine import ACT_CODES
    assert set(_ACTIVATIONS) == set(ao.ACTIVATIONS) == set(a for a in ACT_CODES if a is not None)
    for name in ao.NEW:
        fn = type(name, (), {"__call__": lambda self, x: x})()  # a callable carrying the Keras name
        fn.__name__ = name
        assert Dense(4, activation=name).activation == name
        assert Dense(4, activation=fn).activation == name
        assert LSTMCell(4, activation=name).activation == name
        assert LSTMCell(4, activation=fn).activation == name
        m = DenseSequential(input_dim=3, output_dim=1, num_layers=1, num_units=8, layer_kws=dict(activation=name))
        assert [l.activation for l in m.layers][:-1] == [name, name]
    for bad in ("swish", "gelu"):
        for make in (lambda: Dense(4, activation=bad), lambda: LSTMCell(4, activation=bad),
                     lambda: DenseSequential(input_dim=3, output_dim=1, num_layers=1, num_units=8,
                                             layer_kws=dict(activation=bad))):
            with pytest.raises(ValueError, match="hard_sigmoid"):  # the message lists the accepted names
                make()


def test_plugin_constructors():
    """BORE refuses an activation the kernels do not take when it is built, not at its first proposal."""
    from bore_b200.plugins.hpbandster import BORE
    from bore_b200.plugins.hpbandster._compat import CS
    space = CS.ConfigurationSpace(seed=0)
    space.add_hyperparameter(CS.UniformFloatHyperparameter("x", lower=0.0, upper=1.0))
    for name in ao.NEW:
        assert BORE(space, activation=name).config_generator.activation == name
    for bad in ("swish", "gelu"):
        with pytest.raises(ValueError, match="softplus"):
            BORE(space, activation=bad)


def test_header_enum_matches_act_codes():
    from bore_b200.engine import ACT_CODES
    with open(os.path.join(ROOT, "include", "bore_b200.h")) as fh:
        enum = dict((k.lower(), int(v)) for k, v in re.findall(r"BORE_ACT_([A-Z_]+) = (\d+)", fh.read()))
    assert enum == {k: v for k, v in ACT_CODES.items() if k is not None}


def test_create_range_check(native_lib):
    """Codes 5..9 pass the range check (the call then stops at the device lookup, or succeeds on a
    GPU); -1 and 10 are refused with the message of before, ahead of any device work."""
    lib = native_lib
    dims = (C.c_int * 3)(3, 8, 1)
    for code in range(10):
        h = C.c_void_p()
        rc = lib.bore_mlp_create(2, dims, (C.c_int * 2)(code, 3), 1, 0, C.byref(h))
        msg = lib.bore_last_error().decode()
        if rc == 0:
            lib.bore_mlp_destroy(h)
        else:
            assert "unknown activation" not in msg, (code, msg)
        hl = C.c_void_p()
        rc = lib.bore_lstm_create(3, 8, 1, code, 0, C.byref(hl))
        if rc == 0:
            lib.bore_lstm_destroy(hl)
        else:
            assert "unknown activation" not in lib.bore_last_error().decode(), code
    for code in (-1, 10):
        h = C.c_void_p()
        assert lib.bore_mlp_create(2, dims, (C.c_int * 2)(code, 3), 1, 0, C.byref(h)) != 0
        assert lib.bore_last_error().decode() == f"bore_mlp_create: unknown activation code {code}"
        assert lib.bore_lstm_create(3, 8, 1, code, 0, C.byref(h)) != 0
        assert lib.bore_last_error().decode() == f"bore_lstm_create: unknown activation {code}"
