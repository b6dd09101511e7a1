"""The LSTM kernels (csrc/lstm.cu) across the whole envelope the factory accepts -- input_dim <= 32,
units <= 32, cells <= 4, steps <= 8, batch <= 64 -- against the fp64 oracle (oracle/keras_lstm.py),
with the bars of tests/test_gpu_lstm.py: one unit, odd unit counts, inputs wider than the units (the
fit's [x ; h] rows of the upper cells have a zero tail), one input, the plugin's default net, and the
nets whose BPTT strips do not fit eight warps (the fit then runs fewer sample warps, value and
gradient fewer warps).  Each sample warp keeps T x L x 6 x U floats, so the warp count falls with
steps and cells; from the shared-memory plan of csrc/lstm.cu:

    net (D, U, L, T)   weights    strip    fit sample warps   value-and-gradient warps
    (32, 32, 3, 6)     100,752    15,104   8                  4
    (32, 32, 3, 7)     100,752    17,408   7                  4
    (32, 32, 3, 8)     100,752    19,712   6                  4
    (32, 32, 4, 3)     134,288    10,624   8                  4
    (32, 32, 4, 8)     134,288    25,984   3                  3
    (32, 24, 4, 8)      79,248    19,552   7                  4
    (1, 32, 4, 5)      118,304    16,656   6                  4
    (bytes)

The CPU tests at the end pin that the edges of the envelope are refused before any device work."""
import ctypes as C
import logging

import numpy as np
import pytest

from oracle import keras_lstm as kl
import activation_oracle as ao
from helpers import lstm_factory, lstm_sequences

gpu = pytest.mark.gpu

# name: (D, U, L, activation)
SHAPES = {
    "u1": (3, 1, 1, "tanh"),                 # one unit
    "u1_l4": (1, 1, 4, "sigmoid"),           # one unit, one input, four cells
    "u5": (5, 5, 2, "elu"),
    "u17_softplus": (9, 17, 3, "softplus"),  # extended activation: the EXT builds
    "u31": (31, 31, 1, "relu"),
    "d32_u8": (32, 8, 3, "tanh"),            # D > U: zero tail in the upper cells' [x ; h] rows
    "d1": (1, 16, 2, "elu"),
    "plugin": (32, 32, 2, "elu"),            # the plugin's default cells on a 32-D space
    "l3": (32, 32, 3, "tanh"),               # 8 sample warps up to T = 6, 7 at T = 7, 6 at T = 8
    "l4": (32, 32, 4, "elu"),                # 8 sample warps at T = 3, 3 at T = 8 (and 3 value warps)
    "u24_l4_selu": (32, 24, 4, "selu"),      # 7 sample warps at T = 8
    "d1_l4": (1, 32, 4, "tanh"),             # 6 sample warps at T = 5
}
NAMES = list(SHAPES)
MV = -1.0


@pytest.fixture(autouse=True, scope="module")
def _extended_oracle():
    """the oracle with the extended activations (softplus, selu) of two of the nets"""
    with ao.installed():
        yield


def _bound(ref):
    return 1e-5 * max(1.0, np.abs(ref).max())


def _masked_sequences(seed, N, T, D):
    """lstm_sequences (leading masked steps, gaps, trailing masked steps) with, when N > 2, one sequence
    masked at every step and, at T >= 4, one with two leading masked steps and a gap."""
    X, Y = lstm_sequences(seed, N, T, D, MV)
    if N <= 2:
        return X, Y
    X[N // 2] = MV; Y[N // 2] = MV
    if T >= 4:
        X[1] = np.random.RandomState(seed).uniform(size=(T, D)); Y[1] = 0.0
        X[1, :2] = MV; X[1, 3] = MV; Y[1, :2] = MV; Y[1, 3] = MV
    return X, Y


# ---------------------------------------------------------------- forward
@gpu
@pytest.mark.parametrize("name", NAMES)
def test_forward_with_masking_and_one_to_one(name):
    D, U, L, act = SHAPES[name]
    fac = lstm_factory(D, U, L, act)
    w = kl.init_weights(D, U, L, seed=11)
    net = fac.build_many_to_many(mask_value=MV)
    net.set_weights(w)
    for T in (1, 3, 8):
        X, _ = _masked_sequences(T, 40, T, D)
        mask = kl.compute_mask(X.astype(np.float32), np.float32(MV))
        assert not mask[40 // 2].any() and mask.any()
        got = net.predict(X)
        ref = kl.forward(w, act, X, mask, np.float64)
        assert got.shape == (40, T, 1)
        assert np.abs(got[..., 0] - ref).max() <= _bound(ref), (T, np.abs(got[..., 0] - ref).max())
    for S in (1, 5000):  # 5,000 rows: the grid-stride loop of the forward kernel wraps
        Xs = np.random.RandomState(S).uniform(size=(S, D))
        for T in (1, 3, 8):
            ref = kl.predict_one_to_one(w, act, Xs, T, np.float64)
            got = fac.build_one_to_one(T).predict(Xs)
            assert got.shape == (S, 1) and np.abs(got - ref).max() <= _bound(ref), (S, T)


# ---------------------------------------------------------------- value and input gradient
@gpu
@pytest.mark.parametrize("S", [1, 9, 5000])  # 5,000 points: the grid-stride loop wraps
@pytest.mark.parametrize("name", NAMES)
def test_value_and_input_gradient(name, S):
    import torch
    D, U, L, act = SHAPES[name]
    fac = lstm_factory(D, U, L, act)
    w = kl.init_weights(D, U, L, seed=12)
    net = fac._engine()
    net.set_weights(w)
    X = np.random.RandomState(S + D).uniform(size=(S, D))
    Xd = torch.from_numpy(X.astype(np.float32)).cuda()
    for T in (1, 8):
        for transform in ("identity", "sigmoid", "exp"):
            f64, g64 = kl.value_and_input_grad(w, act, X.astype(np.float32), T, transform, True, np.float64)
            f, g = (a.cpu().numpy() for a in net.value_and_grad_dev(Xd, T, transform, True))
            assert f.shape == (S,) and g.shape == (S, D)
            assert np.abs(f - f64).max() <= _bound(f64), (T, transform, np.abs(f - f64).max())
            assert np.abs(g - g64).max() <= _bound(g64), (T, transform, np.abs(g - g64).max())


@gpu
def test_fp64_points_and_pending_flags_on_three_warps():
    """(32, 32, 4) at 8 steps: value and gradient run 3 warps.  fp64 trial points give what their fp32
    rounding gives, and rows without the pending flag are left alone."""
    import torch
    D, U, L, act = SHAPES["l4"]
    net = lstm_factory(D, U, L, act)._engine()
    net.set_weights(kl.init_weights(D, U, L, seed=13))
    S = 2000
    x64 = torch.from_numpy(np.random.RandomState(4).uniform(size=(S, D))).cuda()
    for transform in ("identity", "sigmoid", "exp"):
        fa, ga = net.value_and_grad_dev(x64, 8, transform, True)
        fb, gb = net.value_and_grad_dev(x64.float(), 8, transform, True)
        assert torch.equal(fa, fb) and torch.equal(ga, gb)
        flags = torch.zeros(S, dtype=torch.int32, device="cuda"); flags[1::3] = 1
        fc = torch.full((S,), -7.0, device="cuda"); gc = torch.full((S, D), -7.0, device="cuda")
        net.value_and_grad_dev(x64, 8, transform, True, flags_dev=flags, f_dev=fc, g_dev=gc)
        on = flags.bool()
        assert torch.equal(fc[on], fa[on]) and torch.equal(gc[on], ga[on])
        assert bool((fc[~on] == -7.0).all()) and bool((gc[~on] == -7.0).all())


# ---------------------------------------------------------------- fit and evaluate
EPOCHS = 6
# (T, N, batch): one step and eight; batch 1, a short last batch (70 = 2 x 32 + 6), batch 64 with a short
# last batch (100 = 64 + 36), batch > N, one sequence
RUNS = [(1, 100, 64), (8, 70, 32), (8, 40, 1), (8, 20, 64), (8, 1, 16)]
FIT_CASES = [(n, T, N, B) for n in NAMES for T, N, B in RUNS]
# either side of the eight-warp boundary of the fit (module docstring)
FIT_CASES += [("l3", 6, 70, 32), ("l3", 7, 70, 32), ("l4", 3, 70, 32), ("d1_l4", 5, 70, 32)]


@gpu
@pytest.mark.parametrize("name,T,N,B", FIT_CASES)
def test_fit_matches_oracle(name, T, N, B):
    """Two fit calls continue one oracle run (the optimizer state persists across fit()), then evaluate."""
    from bore_b200.layers import BinaryCrossentropy
    D, U, L, act = SHAPES[name]
    l2f = 1e-4 if B == 32 else None
    X, Y = _masked_sequences(T * 10 + N, N, T, D)
    rs = np.random.RandomState(5)
    perms = np.stack([rs.permutation(N) for _ in range(EPOCHS)])
    w0 = kl.init_weights(D, U, L, seed=6)
    l2 = None if l2f is None else [l2f, 0, l2f] * L + [0, 0]
    h32, adam32 = kl.fit([a.copy() for a in w0], act, X, Y, EPOCHS, B, perms, MV, l2=l2, dtype=np.float32)
    w64 = [a.astype(np.float64) for a in w0]
    h64, _ = kl.fit(w64, act, X, Y, EPOCHS, B, perms, MV, l2=l2, dtype=np.float64)

    net = lstm_factory(D, U, L, act, l2f=l2f).build_many_to_many(mask_value=MV)
    net.compile(optimizer="adam", loss=BinaryCrossentropy(from_logits=True), metrics=["accuracy"])
    net.set_weights(w0)
    half = EPOCHS // 2
    ha = net.fit(X, Y, epochs=half, batch_size=B, permutations=perms[:half], verbose=0).history["loss"]
    hb = net.fit(X, Y, epochs=EPOCHS - half, batch_size=B, permutations=perms[half:], verbose=0).history["loss"]
    hist = np.array(ha + hb)
    assert np.abs(hist - h64).max() <= 1e-4, (hist, h64)
    assert np.abs(hist - h64).max() <= 4 * max(np.abs(h32 - h64).max(), 2e-6), (hist - h64, h32 - h64)
    for a, b in zip(net.get_weights(), w64):
        assert np.abs(a - b).max() <= 2e-4, np.abs(a - b).max()
    m, v, it = net.get_optimizer_state()
    assert it == adam32.t == EPOCHS * (-(-N // B))
    ev = net.evaluate(X, Y)
    ref = kl.evaluate(w64, act, X, Y, MV, l2=l2, dtype=np.float64)
    live = int(kl.compute_mask(X, MV).sum())
    assert abs(ev[0] - ref[0]) <= 1e-4 and abs(ev[1] - ref[1]) <= 1.5 / max(1, live), (ev, ref)


# ---------------------------------------------------------------- argmax
@gpu
def test_argmax_matches_scipy_on_the_oracle_on_the_largest_net():
    """(32, 32, 4) at 8 steps -- 3 value-and-gradient warps -- against scipy.optimize.minimize(L-BFGS-B)
    driving the oracle, as test_gpu_lstm.py does on a small net: >= 95 % of the starts within 1e-4."""
    from scipy.optimize import Bounds, minimize
    from bore_b200 import ops
    D, U, L, act = SHAPES["l4"]
    T = 8
    X, Y = lstm_sequences(8, 64, T, D, MV)
    Y[..., 0] = np.where(Y[..., 0] < 0, MV, (np.sum((X - 0.4) ** 2, axis=-1) < 2.6).astype(np.float64))
    rs = np.random.RandomState(9)
    perms = np.stack([rs.permutation(64) for _ in range(15)])
    w = kl.init_weights(D, U, L, seed=10)
    kl.fit(w, act, X, Y, 15, 32, perms, MV)
    fac = lstm_factory(D, U, L, act)
    fac.build_many_to_many().set_weights(w)
    one = fac.build_one_to_one(T, transform=ops.sigmoid)
    bounds = Bounds(np.zeros(D), np.ones(D))
    S = 32
    res = one.maxima(bounds, num_starts=S, num_samples=S, print_fn=None, random_state=np.random.RandomState(1))
    X0 = np.random.RandomState(1).uniform(size=(S, D))

    def fn(x):
        f, g = kl.value_and_input_grad(w, act, x[None], T, "sigmoid", True, np.float32)
        return float(f[0]), g[0].astype(np.float64)
    agree = 0
    for i in range(S):
        r = minimize(fn, x0=X0[i], jac=True, method="L-BFGS-B", bounds=bounds, options=dict(maxiter=1000, ftol=1e-9))
        agree += abs(float(res[i].fun) - r.fun) <= 1e-4
        assert np.all(res[i].x >= 0) and np.all(res[i].x <= 1)
    assert agree >= 0.95 * S, agree


# ---------------------------------------------------------------- the plugin end to end
@gpu
def test_bore_hyperband_four_cells_five_rungs():
    """BOREHyperband on a 6-D space with four cells of 32 units and five rungs (eta = 2, budgets 1/16 ... 1):
    the second Hyperband iteration trains the classifier on 5-step sequences, (6, 32, 4, 5), whose fit
    runs 6 sample warps."""
    from bore_b200.plugins.hpbandster import BOREHyperband
    import test_gpu_lstm as tgl
    opt = BOREHyperband(tgl._space(), eta=2, min_budget=1 / 16, max_budget=1, seed=0, num_random_init=1,
                        random_rate=None, num_layers=4, num_units=32, num_steps_per_iter=20, num_starts=2, num_samples=64,
                        logger=logging.getLogger("bore-mf-gpu"))
    cg = opt.config_generator
    steps = []
    fit = cg.logit.fit

    def recording_fit(x, y, **kw):
        steps.append(np.asarray(x).shape[1])
        return fit(x, y, **kw)
    cg.logit.fit = recording_fit
    results = opt.run(n_iterations=2, compute_fn=tgl._loss)
    assert cg.record.num_rungs() == 5 and 5 in steps, steps
    assert 4 in cg.funcs and cg.funcs[4]._last_stats["evals"] > 0
    assert cg.logit.get_optimizer_state()[2] > 0
    assert all(-1.0 <= cfg[f"x{i}"] <= 1.0 for cfg, _, _ in results for i in range(4))


# ---------------------------------------------------------------- the envelope's edges (no GPU needed)
OUTSIDE = [(33, 8, 2, "input_dim=33 outside [1,32]"), (0, 8, 2, "input_dim=0 outside [1,32]"),
           (4, 33, 2, "units=33 outside [1,32]"), (4, 0, 2, "units=0 outside [1,32]"),
           (4, 8, 5, "num_layers=5 outside [1,4]"), (4, 8, 0, "num_layers=0 outside [1,4]")]


@pytest.mark.parametrize("D,U,L,what", OUTSIDE)
def test_create_refuses_outside_the_envelope(native_lib, D, U, L, what):
    from bore_b200.engine import ACT_CODES
    h = C.c_void_p()
    assert native_lib.bore_lstm_create(D, U, L, ACT_CODES["tanh"], 0, C.byref(h)) != 0
    assert native_lib.bore_last_error().decode() == f"bore_lstm_create: {what}"


@pytest.mark.parametrize("D,U,L", [(32, 32, 4), (1, 1, 1), (1, 32, 4), (32, 1, 4)])
def test_create_accepts_the_corners_of_the_envelope(native_lib, D, U, L):
    from bore_b200.engine import ACT_CODES
    h = C.c_void_p()
    rc = native_lib.bore_lstm_create(D, U, L, ACT_CODES["tanh"], 0, C.byref(h))
    if native_lib.bore_device_count() > 0:
        assert rc == 0, native_lib.bore_last_error().decode()
        native_lib.bore_lstm_destroy(h)
    else:  # the envelope check passed and the device check is what refused it
        assert native_lib.bore_last_error().decode() == \
            "bore_lstm_create: no CUDA device visible -- bore_b200 has no CPU fallback"


@pytest.mark.parametrize("D,U,L", [(D, U, L) for D, U, L, _ in OUTSIDE])
def test_factory_refuses_outside_the_envelope(D, U, L):
    from bore_b200.models import StackedRecurrentFactory
    with pytest.raises(NotImplementedError, match="csrc/lstm.cu limits"):
        StackedRecurrentFactory(D, 1, num_layers=L, num_units=U)


def test_fit_refuses_a_batch_above_64():
    from bore_b200.layers import BinaryCrossentropy
    net = lstm_factory(4, 8, 2, "tanh").build_many_to_many(mask_value=MV)
    net.compile(optimizer="adam", loss=BinaryCrossentropy(from_logits=True))
    with pytest.raises(NotImplementedError, match="batch_size <= 64"):
        net.fit(np.zeros((3, 2, 4)), np.zeros((3, 2, 1)), batch_size=65)
