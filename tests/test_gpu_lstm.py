"""LSTM multi-fidelity classifier on the GPU (csrc/lstm.cu, SURVEY.md section 8f row 4) against the
NumPy oracle (oracle/keras_lstm.py, itself checked against torch autograd in tests/test_oracle_lstm.py):
many-to-many logits with masking, the one-to-one network, value + input gradient (1e-5 relative, fp32),
the whole fit (loss trajectory within 1e-4, as north_star asks of training), evaluate, the argmax against
SciPy's L-BFGS-B driving the oracle, and the HpBandSter plugin end to end.  Parity unpinned like the MLP
half: TensorFlow cannot run here (oracle header)."""
import logging

import numpy as np
import pytest

from oracle import keras_lstm as kl
from helpers import lstm_factory as _factory, lstm_sequences as _sequences

pytestmark = pytest.mark.gpu


CASES = [(5, 8, 2, "tanh"), (8, 32, 2, "elu"), (3, 16, 1, "relu"), (32, 32, 3, "elu"), (6, 24, 4, "sigmoid")]


@pytest.mark.parametrize("D,U,L,activation", CASES)
def test_forward_with_masking_and_one_to_one(D, U, L, activation):
    fac = _factory(D, U, L, activation)
    w = kl.init_weights(D, U, L, seed=11)
    for mv in (-1.0, 1e-9):
        X, _ = _sequences(1, 37, 5, D, mv)
        net = fac.build_many_to_many(mask_value=mv)
        net.set_weights(w)
        got = net.predict(X)
        mask = kl.compute_mask(X.astype(np.float32), np.float32(mv))
        assert not mask.all()
        ref = kl.forward(w, activation, X, mask, np.float64)
        assert got.shape == (37, 5, 1)
        assert np.abs(got[..., 0] - ref).max() <= 1e-5 * max(1.0, np.abs(ref).max())
    Xs = np.random.RandomState(2).uniform(size=(50, D))
    for T in (1, 3, 8):
        one = fac.build_one_to_one(T)
        ref = kl.predict_one_to_one(w, activation, Xs, T, np.float64)
        got = one.predict(Xs)
        assert got.shape == (50, 1) and np.abs(got - ref).max() <= 1e-5 * max(1.0, np.abs(ref).max())
    assert [a.shape for a in fac.build_many_to_many().get_weights()] == [a.shape for a in w]
    assert all(np.array_equal(a, b) for a, b in zip(fac.build_many_to_many().get_weights(), w))


@pytest.mark.parametrize("D,U,L,activation", CASES)
@pytest.mark.parametrize("transform", ["identity", "sigmoid", "exp"])
def test_value_and_input_gradient(D, U, L, activation, transform):
    import bore_b200
    from bore_b200 import ops
    fac = _factory(D, U, L, activation)
    w = kl.init_weights(D, U, L, seed=12)
    fac.build_many_to_many().set_weights(w)
    X = np.random.RandomState(3).uniform(size=(64, D))
    for T in (1, 4):
        one = fac.build_one_to_one(T, transform=ops.TRANSFORMS[transform])
        f64, g64 = kl.value_and_input_grad(w, activation, X, T, transform, True, np.float64)
        f, g = one._func_min(X)              # the convert() closure on a batch: [f (S,), g (S, D)]
        assert f.shape == (64,) and g.shape == (64, D) and g.dtype == np.float64
        assert np.abs(f - f64).max() <= 1e-5 * max(1.0, np.abs(f64).max())
        assert np.abs(g - g64).max() <= 1e-5 * max(1.0, np.abs(g64).max())
        f1, g1 = one._func_min(X[7])         # single point: scalar value, (D,) gradient, as a list
        assert np.shape(f1) == () and g1.shape == (D,)
        assert abs(f1 - f[7]) <= 1e-6 * max(1.0, abs(f[7])) and np.abs(g1 - g[7]).max() <= 1e-6 * max(1.0, np.abs(g).max())
    # fp64 trial points (the stepper's buffer) are rounded to fp32 inside the kernel
    import torch
    net = fac._engine()
    x64 = torch.from_numpy(X).cuda()
    fa, ga = net.value_and_grad_dev(x64, 3, transform, True)
    fb, gb = net.value_and_grad_dev(x64.float(), 3, transform, True)
    assert torch.equal(fa, fb) and torch.equal(ga, gb)
    flags = torch.zeros(64, dtype=torch.int32, device="cuda"); flags[::2] = 1
    fc = torch.full((64,), -7.0, device="cuda"); gc = torch.full((64, D), -7.0, device="cuda")
    net.value_and_grad_dev(x64, 3, transform, True, flags_dev=flags, f_dev=fc, g_dev=gc)
    assert torch.equal(fc[::2], fa[::2]) and bool((fc[1::2] == -7.0).all()) and bool((gc[1::2] == -7.0).all())


@pytest.mark.parametrize("D,U,L,activation,N,B,l2f", [
    (5, 8, 2, "tanh", 40, 16, None),
    (8, 32, 2, "elu", 100, 64, 1e-4),      # the plugin's defaults: ragged last batch of 36
    (4, 16, 3, "elu", 70, 32, None),
    (32, 32, 1, "relu", 33, 64, 1e-3),     # one short batch per epoch
])
def test_fit_matches_oracle(D, U, L, activation, N, B, l2f):
    from bore_b200.layers import BinaryCrossentropy
    T, mv, E = 4, -1.0, 12
    X, Y = _sequences(4, N, T, D, mv)
    rs = np.random.RandomState(5)
    perms = np.stack([rs.permutation(N) for _ in range(E)])
    w0 = kl.init_weights(D, U, L, seed=6)
    l2 = None if l2f is None else [l2f, 0, l2f] * L + [0, 0]
    w32 = [a.copy() for a in w0]
    h32, adam32 = kl.fit(w32, activation, X, Y, E, B, perms, mv, l2=l2, dtype=np.float32)
    w64 = [a.astype(np.float64) for a in w0]
    h64, _ = kl.fit(w64, activation, X, Y, E, B, perms, mv, l2=l2, dtype=np.float64)

    fac = _factory(D, U, L, activation, l2f=l2f)
    net = fac.build_many_to_many(mask_value=mv)
    net.compile(optimizer="adam", loss=BinaryCrossentropy(from_logits=True), metrics=["accuracy"])
    net.set_weights(w0)
    half = E // 2                                    # two calls: Adam's state persists across fit()
    ha = net.fit(X, Y, epochs=half, batch_size=B, permutations=perms[:half], verbose=0).history["loss"]
    hb = net.fit(X, Y, epochs=E - half, batch_size=B, permutations=perms[half:], verbose=0).history["loss"]
    hist = np.array(ha + hb)
    assert np.abs(hist - h64).max() <= 1e-4, (hist, h64)          # north_star's training bar
    assert np.abs(hist - h64).max() <= 4 * max(np.abs(h32 - h64).max(), 2e-6)
    got = net.get_weights()
    for a, b in zip(got, w64):
        assert np.abs(a - b).max() <= 2e-4
    m, v, it = net.get_optimizer_state()
    assert it == adam32.t == E * (-(-N // B))
    ev = net.evaluate(X, Y)
    ref = kl.evaluate(w64, activation, X, Y, mv, l2=l2, dtype=np.float64)
    assert abs(ev[0] - ref[0]) <= 1e-4 and abs(ev[1] - ref[1]) <= 1.5 / max(1, int(kl.compute_mask(X, mv).sum()))
    assert hist[-1] < hist[0]


def test_argmax_matches_scipy_on_the_oracle():
    """Every start of the device argmax against scipy.optimize.minimize(L-BFGS-B) driving the oracle's
    value-and-gradient of the same one-to-one network (bore/mixins.py:57-61 with the LSTM model)."""
    from scipy.optimize import Bounds, minimize
    from bore_b200 import ops
    D, U, L, T, activation = 6, 32, 2, 3, "elu"
    # weights with some structure: a short oracle fit on labelled sequences
    X, Y = _sequences(8, 90, T, D, -1.0)
    Y[..., 0] = np.where(Y[..., 0] < 0, -1.0, (np.sum((X - 0.4) ** 2, axis=-1) < 0.45).astype(np.float64))
    rs = np.random.RandomState(9)
    perms = np.stack([rs.permutation(90) for _ in range(40)])
    w = kl.init_weights(D, U, L, seed=10)
    kl.fit(w, activation, X, Y, 40, 32, perms, -1.0)
    fac = _factory(D, U, L, activation)
    fac.build_many_to_many().set_weights(w)
    one = fac.build_one_to_one(T, transform=ops.sigmoid)
    bounds = Bounds(np.zeros(D), np.ones(D))
    S = 96
    res = one.maxima(bounds, num_starts=S, num_samples=S, print_fn=None, random_state=np.random.RandomState(1))
    X0 = np.random.RandomState(1).uniform(size=(S, D))

    def fn(x):
        f, g = kl.value_and_input_grad(w, activation, x[None], T, "sigmoid", True, np.float32)
        return float(f[0]), g[0].astype(np.float64)
    agree = 0
    for i in range(S):
        r = minimize(fn, x0=X0[i], jac=True, method="L-BFGS-B", bounds=bounds, options=dict(maxiter=1000, ftol=1e-9))
        agree += abs(float(res[i].fun) - r.fun) <= 1e-4
        assert np.all(res[i].x >= 0) and np.all(res[i].x <= 1)
    assert agree >= 0.95 * S, agree                   # north_star: >= 95 % of starts agree (smooth ELU net)
    best = one.argmax(bounds, num_starts=S, num_samples=S, print_fn=None, random_state=np.random.RandomState(1))
    ok = [r for r in res if r.success or r.status == 1]
    assert best.fun == min(r.fun for r in ok)
    assert one._last_stats["evals"] >= S
    # screening: 256 samples, the 8 best start (bore/mixins.py:49-56)
    r8 = one.maxima(bounds, num_starts=8, num_samples=256, print_fn=None, random_state=np.random.RandomState(2))
    assert len(r8) == 8
    r0 = one.maxima(bounds, num_starts=0, num_samples=64, print_fn=None, random_state=np.random.RandomState(2))
    assert len(r0) == 1 and r0[0].success


def _space():
    from bore_b200.plugins.hpbandster._compat import CS
    cs = CS.ConfigurationSpace(seed=3)
    for i in range(4):
        cs.add_hyperparameter(CS.UniformFloatHyperparameter(f"x{i}", lower=-1.0, upper=1.0))
    cs.add_hyperparameter(CS.CategoricalHyperparameter("act", ["a", "b"]))
    return cs  # dense dimension 4 + 2 = 6


def _loss(cfg, budget):
    x = np.array([cfg[f"x{i}"] for i in range(4)])
    return np.sum((x - 0.3) ** 2) + (0.2 if cfg["act"] == "a" else 0.0) + 0.05 / budget * np.sin(37.0 * np.sum(x))


def test_bore_hyperband_end_to_end():
    from bore_b200.plugins.hpbandster import BOREHyperband
    opt = BOREHyperband(_space(), eta=3, min_budget=1 / 9, max_budget=1, seed=0, num_random_init=6,
                        num_steps_per_iter=100, num_starts=4, num_samples=128,
                        logger=logging.getLogger("bore-mf-gpu"))
    cg = opt.config_generator
    results = opt.run(n_iterations=6, compute_fn=_loss)
    assert len(results) >= 40
    assert cg.record.num_rungs() == 3 and cg.funcs, "no classifier-driven proposal happened"
    assert all(f._last_stats["evals"] > 0 for f in cg.funcs.values())
    m, v, it = cg.logit.get_optimizer_state()
    assert it > 0
    for cfg, _, _ in results:
        assert cfg["act"] in ("a", "b") and all(-1.0 <= cfg[f"x{i}"] <= 1.0 for i in range(4))
    full = [l for _, b, l in results if b == 1.0]
    assert min(full) < np.mean([l for _, _, l in results[:8]])
