"""The Keras learning-rate schedules ExponentialDecay, InverseTimeDecay, PolynomialDecay and PiecewiseConstantDecay:
the oracle (tests/schedule_oracle.py) against hand-computed values and a float64 restatement, oracle fits against an
independent torch-CPU fit whose rate is set by hand every step, and the host-side surface (classes, refusals, the C
enum and the native argument checks).  CPU only."""
import ctypes as C
import os
import re
import types

import numpy as np
import pytest
import torch

from oracle import keras_lstm as kl, keras_mlp as km
import optimizer_oracle as oo
import schedule_oracle as so
import test_oracle_optimizers as too
from bore_b200 import layers, schedules
from bore_b200.schedules import ExponentialDecay, InverseTimeDecay, PiecewiseConstantDecay, PolynomialDecay

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

# rates that change materially within 100 steps
SCHEDULES = {
    "exponential": lambda: ExponentialDecay(1e-2, 25, 0.5),
    "exponential_staircase": lambda: ExponentialDecay(1e-2, 20, 0.5, staircase=True),
    "inverse_time": lambda: InverseTimeDecay(1e-2, 10, 1.0),
    "inverse_time_staircase": lambda: InverseTimeDecay(1e-2, 15, 2.0, staircase=True),
    "polynomial": lambda: PolynomialDecay(1e-2, 60, end_learning_rate=1e-3, power=2.0),
    "polynomial_cycle": lambda: PolynomialDecay(1e-2, 30, end_learning_rate=1e-3, power=0.5, cycle=True),
    "piecewise": lambda: PiecewiseConstantDecay([20, 50, 80], [1e-2, 5e-3, 2e-3, 1e-3]),
}
# the kinds that take a schedule, one configuration per place the rate enters the rule
KINDS = {
    "adam": lambda lr: layers.Adam(learning_rate=lr),
    "rmsprop": lambda lr: layers.RMSprop(learning_rate=lr),
    "rmsprop_momentum": lambda lr: layers.RMSprop(learning_rate=lr, momentum=0.9),
    "adagrad": lambda lr: layers.Adagrad(learning_rate=lr),
    "adadelta": lambda lr: layers.Adadelta(learning_rate=lr),
    "adamax": lambda lr: layers.Adamax(learning_rate=lr),
}


# ---------------------------------------------------------------------------------------------- the schedules
HAND = [  # (schedule, step, value), computed by hand from the Keras formulas
    (ExponentialDecay(0.1, 10, 0.5), 0, 0.1), (ExponentialDecay(0.1, 10, 0.5), 5, 0.1 * 0.5 ** 0.5),
    (ExponentialDecay(0.1, 10, 0.5), 10, 0.05), (ExponentialDecay(0.1, 10, 0.5), 25, 0.1 * 0.5 ** 2.5),
    (ExponentialDecay(0.1, 10, 0.5, staircase=True), 9, 0.1),
    (ExponentialDecay(0.1, 10, 0.5, staircase=True), 10, 0.05),
    (ExponentialDecay(0.1, 10, 0.5, staircase=True), 19, 0.05),
    (ExponentialDecay(0.1, 10, 0.5, staircase=True), 20, 0.025),
    (InverseTimeDecay(0.1, 10, 1.0), 0, 0.1), (InverseTimeDecay(0.1, 10, 1.0), 10, 0.05),
    (InverseTimeDecay(0.1, 10, 1.0), 5, 0.1 / 1.5), (InverseTimeDecay(0.1, 10, 1.0), 30, 0.025),
    (InverseTimeDecay(0.1, 10, 2.0, staircase=True), 9, 0.1),
    (InverseTimeDecay(0.1, 10, 2.0, staircase=True), 10, 0.1 / 3),
    (InverseTimeDecay(0.1, 10, 2.0, staircase=True), 29, 0.1 / 5),
    (PolynomialDecay(0.1, 10, 0.01), 0, 0.1), (PolynomialDecay(0.1, 10, 0.01), 5, 0.055),
    (PolynomialDecay(0.1, 10, 0.01), 10, 0.01), (PolynomialDecay(0.1, 10, 0.01), 25, 0.01),  # clamped
    (PolynomialDecay(0.1, 10, 0.01, power=2.0), 5, 0.0325), (PolynomialDecay(0.1, 10), 10, 1e-4),
    (PolynomialDecay(0.1, 10, 0.01, cycle=True), 0, 0.1),  # ceil(0) would be 0: the multiplier is 1
    (PolynomialDecay(0.1, 10, 0.01, cycle=True), 5, 0.055),
    (PolynomialDecay(0.1, 10, 0.01, cycle=True), 10, 0.01),  # multiple of decay_steps: the end of a cycle
    (PolynomialDecay(0.1, 10, 0.01, cycle=True), 11, 0.09 * 0.45 + 0.01),  # decay_steps 20
    (PolynomialDecay(0.1, 10, 0.01, cycle=True), 20, 0.01),
    (PolynomialDecay(0.1, 10, 0.01, cycle=True), 21, 0.09 * 0.3 + 0.01),  # decay_steps 30
    (PiecewiseConstantDecay([10, 20], [1.0, 0.5, 0.1]), 0, 1.0),
    (PiecewiseConstantDecay([10, 20], [1.0, 0.5, 0.1]), 10, 1.0),
    (PiecewiseConstantDecay([10, 20], [1.0, 0.5, 0.1]), 11, 0.5),
    (PiecewiseConstantDecay([10, 20], [1.0, 0.5, 0.1]), 20, 0.5),
    (PiecewiseConstantDecay([10, 20], [1.0, 0.5, 0.1]), 21, 0.1),
    (PiecewiseConstantDecay([10], [1e-3, 0.0]), 10, 1e-3), (PiecewiseConstantDecay([10], [1e-3, 0.0]), 11, 0.0),
    (PiecewiseConstantDecay([10.5], [1.0, 2.0]), 10, 1.0), (PiecewiseConstantDecay([10.5], [1.0, 2.0]), 11, 2.0),
]


@pytest.mark.parametrize("i", range(len(HAND)))
def test_hand_values(i):
    s, step, want = HAND[i]
    got = so.rate(s)(step)
    assert isinstance(got, np.float32)
    assert got == pytest.approx(want, rel=2e-7, abs=0), (s.get_config(), step)
    assert s(step) == got  # the class's own __call__: the same float32


@pytest.mark.parametrize("name", sorted(SCHEDULES))
def test_float32_against_float64(name):
    """The float32 arithmetic rounds each operation: it stays within float32 rounding of float64 over the steps of
    a long run (2e-6 relative: pow amplifies the rounding of its exponent p by |p ln(decay_rate)|, 11 at most
    here)."""
    s = SCHEDULES[name]()
    kind = {"ExponentialDecay": "exponential", "InverseTimeDecay": "inverse_time", "PolynomialDecay": "polynomial",
            "PiecewiseConstantDecay": "piecewise"}[type(s).__name__]
    fn = so.rate(s)
    for step in range(0, 400):
        got, want = fn(step), so.exact(step, kind, **s.get_config())
        assert abs(float(got) - want) <= 2e-6 * abs(want), (step, got, want)
        assert s(step) == got


def test_piecewise_boundaries_compare_in_float32():
    """TF casts the boundaries and the step to float32: 2^24 + 1 becomes 2^24, so step 2^24 is not past it, and
    step 2^24 + 5 becomes 2^24 + 4, the second boundary.  The native parameters carry the float32 boundaries."""
    s = PiecewiseConstantDecay([2 ** 24 + 1, 2 ** 24 + 4], [1.0, 0.5, 0.25])
    assert so.rate(s)(2 ** 24) == s(2 ** 24) == np.float32(1.0)
    assert s(2 ** 24 + 2) == s(2 ** 24 + 5) == np.float32(0.5) and s(2 ** 24 + 6) == np.float32(0.25)
    assert s.native() == (4, [2.0 ** 24, 2.0 ** 24 + 4, 1.0, 0.5, 0.25])


# ---------------------------------------------------------------------------------------------- oracle fits
def _torch_fit(w0, loss_fn, N, epochs, batch, perms, o, l2):
    """test_oracle_optimizers' torch fit with the rate of update t set by hand to the schedule at t - 1."""
    fn = so.rate(o.learning_rate)
    spec = types.SimpleNamespace(**dict(vars(o), learning_rate=float(fn(0))), kind=o.kind)
    ws = [torch.tensor(a, requires_grad=True) for a in w0]
    opt = too.torch_optimizer(ws, spec)
    hist, t = [], 0
    for e in range(epochs):
        tot = 0.0
        for s in range(0, N, batch):
            idx = torch.as_tensor(perms[e][s:s + batch])
            loss = loss_fn(ws, idx) + sum(l2 * (a * a).sum() for a in ws)
            opt.zero_grad()
            loss.backward()
            spec.learning_rate = float(fn(t))  # _Hand reads the spec, torch.optim the group
            for g in opt.param_groups:
                g["lr"] = spec.learning_rate
            opt.step()
            t += 1
            tot += float(loss.detach()) * len(idx)
        hist.append(tot / N)
    return np.array(hist), [a.detach().numpy() for a in ws]


MLP_CASES = [(s, k, 0) for s in sorted(SCHEDULES) for k in sorted(KINDS)] + \
            [(s, k, 1) for s in sorted(SCHEDULES) for k in ("adam", "rmsprop_momentum")]
NETS = [([4, 16, 8, 1], ["elu", "tanh", "sigmoid"], 0.0), ([3, 12, 1], ["relu", "linear"], 1e-3)]


@pytest.mark.parametrize("sched,kind,net", MLP_CASES)
def test_mlp_fit_vs_torch(sched, kind, net):
    """100 steps (25 epochs x 4 batches) of the oracle fit loop under the kind's rule and the schedule."""
    dims, acts, l2 = NETS[net]
    o = KINDS[kind](SCHEDULES[sched]())
    rs = np.random.RandomState(3)
    N, E, B = 100, 25, 25
    X = rs.uniform(-1.5, 1.5, size=(N, dims[0]))
    y = np.sum((X - 0.3) ** 2, axis=1)
    z = (y < np.quantile(y, 0.3)).astype(np.float64)
    perms = np.stack([rs.permutation(N) for _ in range(E)])
    w0 = km.init_weights(dims, 5, np.float64)
    w = [a.copy() for a in w0]
    with oo.installed(), so.installed(o.learning_rate):
        hist, st = km.fit(w, acts, X, z, E, B, perms, adam=oo.state_for(w, o, np.float64), l2=l2,
                          dtype=np.float64)
    assert st.t == 100
    Xt, zt = torch.tensor(X), torch.tensor(z).reshape(-1, 1)
    bce = torch.nn.functional.binary_cross_entropy_with_logits
    hist_t, wt = _torch_fit(w0, lambda ws, idx: bce(too._torch_mlp(ws, acts, Xt[idx]), zt[idx]), N, E, B, perms,
                            o, l2)
    assert np.abs(hist - hist_t).max() <= 1e-10
    assert max(np.abs(a - b).max() for a, b in zip(w, wt)) <= 1e-10


@pytest.mark.parametrize("sched", sorted(SCHEDULES))
@pytest.mark.parametrize("kind", ["adam", "adagrad", "rmsprop_momentum"])
def test_lstm_fit_vs_torch(sched, kind):
    """100 steps (50 epochs x 2 batches) of keras_lstm's fit loop under the kind's rule and the schedule."""
    o = KINDS[kind](SCHEDULES[sched]())
    D, U, L, T, N, E, B = 4, 8, 2, 3, 40, 50, 20
    rs = np.random.RandomState(7)
    X = rs.uniform(size=(N, T, D))
    Y = (rs.uniform(size=(N, T, 1)) < 0.4).astype(np.float64)
    perms = np.stack([rs.permutation(N) for _ in range(E)])
    w0 = kl.init_weights(D, U, L, seed=8, dtype=np.float64)
    w = [a.copy() for a in w0]
    with oo.installed(), so.installed(o.learning_rate):
        hist, st = kl.fit(w, "tanh", X, Y, E, B, perms, mask_value=-1e9, adam=oo.state_for(w, o, np.float64),
                          dtype=np.float64)
    assert st.t == 100
    Xt, Yt = torch.tensor(X), torch.tensor(Y[..., 0])
    bce = torch.nn.functional.binary_cross_entropy_with_logits
    hist_t, wt = _torch_fit(w0, lambda ws, idx: bce(too._torch_lstm(ws, Xt[idx]), Yt[idx]), N, E, B, perms, o, 0.0)
    assert np.abs(hist - hist_t).max() <= 1e-10
    assert max(np.abs(a - b).max() for a, b in zip(w, wt)) <= 1e-10


def test_schedule_changes_the_fit():
    """The hook is live: the same fit under a constant rate ends elsewhere."""
    dims, acts, _ = NETS[0]
    rs = np.random.RandomState(3)
    X = rs.uniform(-1.5, 1.5, size=(100, 4))
    z = (np.sum(X ** 2, axis=1) < 1.5).astype(np.float32)
    perms = np.stack([rs.permutation(100) for _ in range(10)])
    out = []
    for lr in (1e-2, PiecewiseConstantDecay([10], [1e-2, 1e-3])):
        o = layers.Adam(learning_rate=lr)
        w = km.init_weights(dims, 5)
        with so.installed(o.learning_rate) if lr != 1e-2 else oo.installed():
            km.fit(w, acts, X, z, 10, 25, perms, adam=oo.state_for(w, layers.Adam(learning_rate=1e-2)))
        out.append(w)
    assert max(np.abs(a - b).max() for a, b in zip(*out)) > 1e-4


# ---------------------------------------------------------------------------------------------- the surface
def test_classes_configs_and_optimizers():
    assert layers.schedules is schedules
    s = PolynomialDecay(0.1, 10)
    assert s.get_config() == {"initial_learning_rate": 0.1, "decay_steps": 10, "end_learning_rate": 0.0001,
                              "power": 1.0, "cycle": False, "name": None}
    for make in SCHEDULES.values():
        a = make()
        b = type(a)(**a.get_config())
        assert all(a(k) == b(k) for k in range(0, 120, 7))
    assert ExponentialDecay(1e-2, 10, 0.9).get_config()["staircase"] is False
    assert InverseTimeDecay(1e-2, 10, 0.9, name="x").get_config()["name"] == "x"
    # an optimizer keeps the schedule as its learning_rate, as Keras does
    for make_opt in KINDS.values():
        sch = ExponentialDecay(1e-2, 10, 0.9)
        o = make_opt(sch)
        assert o.learning_rate is sch and layers.optimizer_spec(o) is o
        code, hp = o.hyper()
        assert hp[0] == 1.0 and o.lr_schedule() == (1, [1e-2, 10.0, 0.9, 0.0])
    # a constant rate: hyper() as before, and the constant schedule
    assert layers.Adam().hyper() == (0, [1e-3, 0.9, 0.999, 1e-7, 0.0, 0.0, 0.0])
    assert layers.Adagrad(learning_rate=0.5).hyper()[1][0] == 0.5
    assert layers.RMSprop().lr_schedule() == (0, [])
    assert PolynomialDecay(1e-2, 30, 1e-3, 0.5, cycle=True).native() == (3, [1e-2, 30.0, 1e-3, 0.5, 1.0])
    assert InverseTimeDecay(1e-2, 15, 2.0, staircase=True).native() == (2, [1e-2, 15.0, 2.0, 1.0])
    assert PiecewiseConstantDecay([20, 50], [1.0, 0.5, 0.25]).native() == (4, [20.0, 50.0, 1.0, 0.5, 0.25])


def test_refusals():
    with pytest.raises(NotImplementedError, match="schedule"):
        layers.Adam(learning_rate=lambda step: 1e-3)

    class Warm(ExponentialDecay):
        def __call__(self, step):
            return min(1.0, step / 10) * super().__call__(step)

    class Mine(schedules.LearningRateSchedule):
        def __call__(self, step):
            return 1e-3

    for s in (Warm(1e-2, 10, 0.9), Mine()):
        with pytest.raises(NotImplementedError, match="schedule"):
            layers.Adagrad(learning_rate=s)
    with pytest.raises(ValueError, match="Nadam"):
        layers.Nadam(learning_rate=ExponentialDecay(1e-2, 10, 0.9))
    with pytest.raises(ValueError, match="1 less"):
        PiecewiseConstantDecay([1, 2], [1.0, 0.5])
    bad = [(ExponentialDecay(1e-2, 0, 0.9), "decay_steps"), (InverseTimeDecay(1e-2, -3, 0.9), "decay_steps"),
           (PolynomialDecay(1e-2, 0), "decay_steps"), (ExponentialDecay(float("nan"), 10, 0.9), "finite"),
           (PolynomialDecay(1e-2, 10, power=float("inf")), "finite"),
           (PiecewiseConstantDecay([5, 5], [1.0, 0.5, 0.25]), "increasing"),
           (PiecewiseConstantDecay([], [1.0]), "boundaries"),
           (PiecewiseConstantDecay(list(range(17)), [1.0] * 18), "boundaries"),
           (PiecewiseConstantDecay([1, 2], [1.0, float("inf"), 0.5]), "finite")]
    for s, what in bad:
        with pytest.raises(ValueError, match=what):
            layers.Adam(learning_rate=s)
    assert layers.Adam(learning_rate=PiecewiseConstantDecay(list(range(16)), [1.0] * 17))


def test_both_surfaces_and_plugins_accept_a_schedule():
    from bore_b200.layers import BinaryCrossentropy, Dense
    from bore_b200.models import MaximizableSequential, StackedRecurrentFactory
    from bore_b200.plugins.hpbandster import BORE, BOREHyperband
    from bore_b200.plugins.hpbandster._compat import CS
    r = MaximizableSequential()
    r.add(Dense(16, activation="relu")); r.add(Dense(1, activation="sigmoid"))
    r.compile(optimizer=layers.RMSprop(learning_rate=InverseTimeDecay(1e-2, 10, 1.0)), loss="binary_crossentropy")
    net = StackedRecurrentFactory(4, 1, num_layers=2, num_units=8).build_many_to_many(mask_value=-1.0)
    net.compile(optimizer=layers.Adam(learning_rate=ExponentialDecay(1e-2, 10, 0.9)),
                loss=BinaryCrossentropy(from_logits=True))
    space = CS.ConfigurationSpace(seed=0)
    space.add_hyperparameter(CS.UniformFloatHyperparameter("x", lower=0.0, upper=1.0))
    for cls in (BORE, BOREHyperband):
        opt = layers.Adam(learning_rate=ExponentialDecay(1e-2, 10, 0.9))
        assert cls(space, optimizer=opt).config_generator.optimizer is opt


def test_header_enum_matches_codes():
    with open(os.path.join(ROOT, "include", "bore_b200.h")) as fh:
        text = fh.read()
    enum = dict((k.lower(), int(v)) for k, v in re.findall(r"BORE_LR_([A-Z_]+) = (\d+)", text))
    assert enum == schedules.LR_CODES
    assert int(re.search(r"#define BORE_LR_MAX_BOUNDARIES (\d+)", text).group(1)) == schedules.MAX_BOUNDARIES
    assert {c.code for c in schedules.SCHEDULES} == set(schedules.LR_CODES.values()) - {0}


def test_native_argument_checks(native_lib):
    """bore_{mlp,lstm}_set_lr_schedule check the kind and the parameters before the handle (no device needed)."""
    lib = native_lib

    def call(fn, kind, sp, n=None):
        arr = (C.c_float * max(1, len(sp)))(*sp)
        rc = getattr(lib, fn)(None, kind, arr, len(sp) if n is None else n)
        return rc, lib.bore_last_error().decode()

    good = [(0, [])] + [make().native() for make in SCHEDULES.values()] + \
        [PiecewiseConstantDecay(list(range(16)), [1.0] * 17).native(), PiecewiseConstantDecay([3], [0.0, 1.0]).native()]
    bad = [(5, [], "unknown schedule kind 5"), (-1, [], "unknown schedule kind -1"),
           (0, [1.0], "takes 0"), (1, [1e-2, 10, 0.9], "takes 4"), (3, [1e-2, 10, 1e-4, 1.0], "takes 5"),
           (1, [1e-2, 0.0, 0.9, 0], "decay_steps"), (2, [1e-2, -1.0, 0.9, 0], "decay_steps"),
           (3, [1e-2, 0.0, 1e-4, 1.0, 0], "decay_steps"), (1, [1e-2, 10, 0.9, 0.5], "staircase"),
           (3, [1e-2, 10, 1e-4, 1.0, 2], "cycle"), (1, [float("nan"), 10, 0.9, 0], "parameter 0"),
           (3, [1e-2, 10, 1e-4, float("inf"), 0], "parameter 3"), (2, [1e-2, float("inf"), 0.9, 0], "parameter 1"),
           (4, [5.0, 5.0, 1.0, 0.5, 0.25], "strictly increasing"), (4, [6.0, 5.0, 1.0, 0.5, 0.25], "strictly"),
           (4, [5.0, 1.0, 0.5, 0.25], "n + 1 values"), (4, [1.0], "n + 1 values"),
           (4, list(range(17)) + [1.0] * 18, "n + 1 values"), (4, [5.0, 1.0, float("nan")], "parameter 2")]
    for fn in ("bore_mlp_set_lr_schedule", "bore_lstm_set_lr_schedule"):
        for code, sp in good:
            rc, msg = call(fn, code, sp)
            assert rc != 0 and msg == "NULL handle", (code, sp, msg)  # every check passed
        for code, sp, what in bad:
            rc, msg = call(fn, code, sp)
            assert rc != 0 and what in msg, (code, sp, msg)
        rc = getattr(lib, fn)(None, 1, None, 4)
        assert rc != 0 and "NULL" in lib.bore_last_error().decode()
        rc = getattr(lib, fn)(None, 0, None, 0)
        assert rc != 0 and lib.bore_last_error().decode() == "NULL handle"
