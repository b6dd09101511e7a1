"""The activations selu, softplus, softsign, hard_sigmoid and exponential on the device, against the oracle
(tests/activation_oracle.py) with the bars of the existing parity tests: K0 / K2, every fit kernel, the
argmax paths (fused, rounds, handover; SciPy), SVGD, the LSTM kernels and both plugins end to end."""
import logging

import numpy as np
import pytest

from oracle import keras_mlp as km, svgd as osv
import activation_oracle as ao
import weighted_oracle as wo
from helpers import synthetic_targets, reference_self_agreement, parallel_minimize_starts

pytestmark = pytest.mark.gpu

RTOL, ATOL = 1e-5, 2e-6
LOSS_TOL = 1e-4

NETS = {
    "selu": ([6, 32, 32, 1], ["selu", "selu", "linear"], "sigmoid"),
    "softplus": ([6, 32, 32, 1], ["softplus", "softplus", "sigmoid"], "identity"),
    "softsign": ([5, 24, 40, 1], ["softsign", "softsign", "linear"], "exp"),
    "hard_sigmoid": ([4, 16, 16, 1], ["hard_sigmoid", "hard_sigmoid", "sigmoid"], "identity"),
    "exponential": ([3, 16, 8, 1], ["tanh", "exponential", "linear"], "sigmoid"),
    "mixed": ([8, 64, 48, 32, 1], ["selu", "softplus", "softsign", "linear"], "sigmoid"),
    "out_softplus": ([4, 16, 1], ["elu", "softplus"], "identity"),       # a new OUTPUT activation
    "out_hard_sigmoid": ([4, 16, 1], ["relu", "hard_sigmoid"], "identity"),
}


@pytest.fixture(autouse=True, scope="module")
def _extended_oracle():
    with ao.installed():
        yield


def _fit_acts(acts):
    return list(acts[:-1]) + ["sigmoid" if acts[-1] == "sigmoid" else "linear"]


def _weights(dims, acts, seed):
    """Glorot init + a short oracle fit: non-degenerate weights."""
    rs = np.random.RandomState(seed)
    w = km.init_weights(dims, seed)
    X = rs.uniform(size=(300, dims[0]))
    y = synthetic_targets(X)
    km.fit(w, _fit_acts(acts), X, y < np.quantile(y, 0.25), 20, 64, [rs.permutation(300) for _ in range(20)])
    return w


def _net(dims, acts, w=None, n_models=1):
    from bore_b200.engine import NativeMLP
    net = NativeMLP(dims, acts, n_models=n_models)
    if w is not None:
        net.set_weights(w)
    return net


@pytest.mark.parametrize("name", sorted(NETS))
@pytest.mark.parametrize("S", [1, 17, 1037])
def test_value_grad_and_predict(name, S):
    dims, acts, _ = NETS[name]
    w = _weights(dims, acts, 1)
    X = np.random.RandomState(S).uniform(-0.2, 1.2, size=(S, dims[0]))
    net = _net(dims, acts, w)
    y, y32 = net.predict(X), km.predict(w, acts, X)
    assert np.all(np.abs(y - y32) <= RTOL * np.abs(y32) + ATOL)
    for transform in ("identity", "sigmoid", "exp"):
        for negate in (True, False):
            f, g = net.value_and_grad(X, transform, negate)
            f32, g32 = km.value_and_input_grad(w, acts, X, transform, negate, np.float32)
            g64 = km.value_and_input_grad(w, acts, X, transform, negate, np.float64)[1]
            gscale = np.abs(g64).max(axis=1, keepdims=True)
            assert np.all(np.abs(f - f32) <= RTOL * np.abs(f32) + ATOL), np.abs(f - f32).max()
            assert np.all(np.abs(g - g32) <= RTOL * gscale + ATOL), (np.abs(g - g32) / (gscale + 1e-30)).max()


def _problem(dims, N, E, seed):
    rs = np.random.RandomState(seed)
    X = rs.uniform(size=(N, dims[0]))
    y = synthetic_targets(X)
    return X, y < np.quantile(y, 0.25), np.stack([rs.permutation(N) for _ in range(E)])


FIT_NETS = ["selu", "softplus", "softsign", "hard_sigmoid", "exponential", "mixed"]


@pytest.mark.parametrize("mode", [1, 2, 3, 4])
@pytest.mark.parametrize("name", FIT_NETS)
@pytest.mark.parametrize("l2", [0.0, 1e-3])
def test_fit_modes(name, mode, l2):
    dims, acts, _ = NETS[name]
    acts = _fit_acts(acts)
    N, E = 333, 12
    X, z, perms = _problem(dims, N, E, seed=5)
    w0 = km.init_weights(dims, 3)
    w_ref = [a.copy() for a in w0]
    h_ref, adam = km.fit(w_ref, acts, X, z, E, 64, perms, l2=l2)
    net = _net(dims, acts, w0)
    net.set_fit_mode(mode)
    hist = net.fit(X, z, E, 64, perms, l2=l2)
    assert np.abs(hist - h_ref).max() <= LOSS_TOL, np.abs(hist - h_ref).max()
    for a, b in zip(net.get_weights(), w_ref):
        assert np.abs(a - b).max() <= 2e-3


@pytest.mark.parametrize("dims,act", [([50, 64, 64, 64, 1], "selu"), ([6, 32, 32, 1], "softplus"),
                                      ([6, 16, 16, 1], "hard_sigmoid"), ([7, 24, 40, 1], "softsign")])
def test_unit_split_builds(dims, act):
    """Fit mode 4: uniform hidden widths 16 / 32 / 64 take the compile-time builds of the unit-split kernel,
    24 / 40 its run-time build."""
    acts = [act] * (len(dims) - 2) + ["sigmoid"]
    N, E = 700, 4
    X, z, perms = _problem(dims, N, E, seed=9)
    w0 = km.init_weights(dims, 4)
    w_ref = [a.copy() for a in w0]
    h_ref, _ = km.fit(w_ref, acts, X, z, E, 64, perms)
    net = _net(dims, acts, w0)
    net.set_fit_mode(4)
    assert np.abs(net.fit(X, z, E, 64, perms) - h_ref).max() <= LOSS_TOL


@pytest.mark.parametrize("M", [20, 600])
def test_many_models(M):
    dims, acts = [6, 32, 32, 1], ["softsign", "selu", "linear"]
    N, E = 150, 6
    probs = [_problem(dims, N, E, seed=50 + i) for i in range(M)]
    ws = [km.init_weights(dims, 200 + i) for i in range(M)]
    net = _net(dims, acts, n_models=M)
    for i, w in enumerate(ws):
        net.set_weights(w, model=i)
    Xd = net.to_device(np.concatenate([p[0] for p in probs]), np.float32)
    zd = net.to_device(np.concatenate([p[1] for p in probs]).astype(np.float32), np.float32)
    pd = net.to_device(np.stack([p[2] for p in probs]).astype(np.int32), np.int32)
    loss = net.fit_dev(Xd, zd, N, 64, E, pd, model0=0, count=M, shared_data=False, shared_perm=False).cpu().numpy()
    for i in list(range(0, M, max(1, M // 25))) + [M - 1]:
        w_ref = [a.copy() for a in ws[i]]
        h_ref, _ = km.fit(w_ref, acts, probs[i][0], probs[i][1], E, 64, probs[i][2])
        assert np.abs(loss[i] - h_ref).max() <= LOSS_TOL, i


def test_weighted_fit():
    dims, acts = [6, 32, 32, 1], ["softplus", "hard_sigmoid", "sigmoid"]
    N, E = 200, 10
    X, z, perms = _problem(dims, N, E, seed=11)
    sw = np.random.RandomState(12).uniform(0, 2, size=N).astype(np.float32)
    w0 = km.init_weights(dims, 6)
    w_ref = [a.copy() for a in w0]
    h_ref, _ = wo.fit(w_ref, acts, X, z, E, 64, perms, sample_weight=sw, class_weight={0: 0.5, 1: 2.0})
    for mode in (1, 2, 4):
        net = _net(dims, acts, w0)
        net.set_fit_mode(mode)
        hist = net.fit(X, z, E, 64, perms, w=sw, class_weight=(0.5, 2.0))
        assert np.abs(hist - h_ref).max() <= LOSS_TOL, mode


def test_ragged_fit():
    from bore_b200.ragged import RaggedLayout
    dims, acts = [5, 32, 32, 1], ["selu", "softsign", "linear"]
    n, e = np.array([40, 130, 75]), np.array([9, 3, 5])
    lay = RaggedLayout(n, e)
    probs = [_problem(dims, int(n[p]), int(e[p]), seed=20 + p) for p in range(3)]
    ws = [km.init_weights(dims, 30 + p) for p in range(3)]
    net = _net(dims, acts, n_models=3)
    for p, w in enumerate(ws):
        net.set_weights(w, model=p)
    Xd = net.to_device(np.concatenate([p[0] for p in probs]), np.float32)
    zd = net.to_device(np.concatenate([p[1] for p in probs]).astype(np.float32), np.float32)
    pd = net.to_device(np.concatenate([p[2].reshape(-1) for p in probs]).astype(np.int32), np.int32)
    loss = net.fit_ragged_dev(Xd, zd, lay, 64, pd).cpu().numpy()
    for p in range(3):
        h_ref, _ = km.fit([a.copy() for a in ws[p]], acts, probs[p][0], probs[p][1], int(e[p]), 64, probs[p][2])
        assert np.abs(loss[lay.losses[p]:lay.losses[p + 1]] - h_ref).max() <= LOSS_TOL, p


KEYS = ("x", "fun", "nit", "nfev", "status", "task")


def _lbfgsb(net, X0, transform, mode, multi=False):
    import torch
    from bore_b200 import _lib
    _lib.check(_lib.require_cuda().bore_lbfgsb_set_mode(mode))
    try:
        net._work = None
        run = net.lbfgsb_multi_dev if multi else net.lbfgsb_dev
        r = run(torch.from_numpy(X0).cuda(), 0.0, 1.0, transform=transform)
    finally:
        _lib.check(_lib.require_cuda().bore_lbfgsb_set_mode(0))
    return {k: (v.cpu().numpy() if hasattr(v, "cpu") else v) for k, v in r.items()}


@pytest.mark.parametrize("name", sorted(NETS))
def test_fused_equals_rounds(name):
    dims, acts, transform = NETS[name]
    net = _net(dims, acts, _weights(dims, acts, 5))
    X0 = np.random.RandomState(7).uniform(size=(700, dims[0]))
    a, b = _lbfgsb(net, X0, transform, 2), _lbfgsb(net, X0, transform, 1)
    assert a["rounds"] == 1 and b["rounds"] > 1
    for k in KEYS:
        assert np.array_equal(a[k], b[k]), k


@pytest.mark.parametrize("name", ["softplus", "selu"])
def test_handover_equals_rounds(name):
    dims, acts, transform = NETS[name]
    net = _net(dims, acts, _weights(dims, acts, 4))
    X0 = np.random.RandomState(11).uniform(size=(20000, dims[0]))
    a, b = _lbfgsb(net, X0, transform, 0), _lbfgsb(net, X0, transform, 1)
    assert 1 < a["rounds"] < b["rounds"]
    for k in KEYS:
        assert np.array_equal(a[k], b[k]), k


def test_batched_argmax_fused_equals_rounds():
    dims, acts = [6, 32, 32, 1], ["softplus", "softsign", "sigmoid"]
    M, K = 23, 5
    net = _net(dims, acts, n_models=M)
    for p in range(M):
        net.set_weights(_weights(dims, acts, 100 + p), model=p)
    X0 = np.random.RandomState(5).uniform(size=(M, K, 6))
    a, b = _lbfgsb(net, X0, "identity", 2, multi=True), _lbfgsb(net, X0, "identity", 1, multi=True)
    for k in KEYS:
        assert np.array_equal(a[k], b[k]), k


@pytest.mark.parametrize("name", ["softplus", "softsign", "selu", "hard_sigmoid"])
def test_argmax_vs_scipy(name):
    """64 starts: smooth nets agree with SciPy on >= 0.99 of them; selu and hard_sigmoid (kinks) are held
    to the reference's own agreement with itself after an fp32 re-association."""
    dims, acts, transform = NETS[name]
    w = _weights(dims, acts, 8)
    X0 = np.random.RandomState(13).uniform(size=(64, dims[0]))
    net = _net(dims, acts, w)
    got = _lbfgsb(net, X0, transform, 0)
    ref = parallel_minimize_starts(w, acts, X0, 0.0, 1.0, transform)
    tol = 1e-4 * max(1.0, float(np.abs(ref["fun"]).max()))
    agree = float(np.mean(np.abs(got["fun"] - ref["fun"]) <= tol))
    if name in ("softplus", "softsign"):
        assert agree >= 0.99, agree
    else:
        from scipy.optimize import Bounds
        self_agree, _, _ = reference_self_agreement(w, acts, X0, Bounds(np.zeros(dims[0]), np.ones(dims[0])),
                                                    transform, tol, ref=ref)
        assert agree >= self_agree - 1 / 64, (agree, self_agree)


def test_svgd_softplus():
    from bore_b200.models import BatchMaximizableSequential
    from bore_b200.layers import Dense
    from bore_b200 import ops
    dims, acts = [6, 32, 32, 1], ["softplus", "softplus", "sigmoid"]
    w = _weights(dims, acts, 3)
    bm = BatchMaximizableSequential(transform=ops.identity)
    for i, (u, a) in enumerate(zip(dims[1:], acts)):
        bm.add(Dense(u, activation=a, input_dim=6 if i == 0 else None))
    bm.compile(optimizer="adam", loss="binary_crossentropy")
    bm.set_weights(w)
    xb = bm.argmax_batch(batch_size=8, bounds=[(0., 1.)] * 6, n_iter=30, random_state=3)
    xr = osv.argmax_batch(w, acts, 8, [(0., 1.)] * 6, n_iter=30, random_state=3)
    assert np.abs(xb - xr).max() <= 1e-4


@pytest.mark.parametrize("activation", ["softplus", "selu", "softsign", "hard_sigmoid"])
def test_lstm(activation):
    import test_gpu_lstm as tgl
    tgl.test_forward_with_masking_and_one_to_one(5, 8, 2, activation)
    tgl.test_value_and_input_gradient(5, 8, 2, activation, "sigmoid")
    tgl.test_fit_matches_oracle(8, 32, 2, activation, 100, 64, 1e-4)


def test_bore_selu_end_to_end():
    import test_gpu_plugin as tgp
    from bore_b200.plugins.hpbandster import BORE
    opt = BORE(tgp._space(), eta=3, min_budget=1 / 9, max_budget=1, seed=0, num_random_init=8,
               num_steps_per_iter=200, num_starts=4, num_samples=256, activation="selu",
               logger=logging.getLogger("bore-test"))
    results = opt.run(n_iterations=4, compute_fn=tgp._loss)
    cg = opt.config_generator
    assert cg.logit is not None and cg.logit._last_stats["evals"] > 0
    assert [l.activation for l in cg.logit.layers][:-1] == ["selu"] * (len(cg.logit.layers) - 1)
    assert min(l for _, b, l in results if b == 1.0) < np.mean([l for _, _, l in results[:8]])


def test_bore_hyperband_softplus_end_to_end():
    import test_gpu_lstm as tgl
    from bore_b200.plugins.hpbandster import BOREHyperband
    opt = BOREHyperband(tgl._space(), eta=3, min_budget=1 / 9, max_budget=1, seed=0, num_random_init=6,
                        num_steps_per_iter=100, num_starts=4, num_samples=128, activation="softplus",
                        logger=logging.getLogger("bore-mf-gpu"))
    cg = opt.config_generator
    results = opt.run(n_iterations=6, compute_fn=tgl._loss)
    assert cg.funcs and all(f._last_stats["evals"] > 0 for f in cg.funcs.values())
    assert min(l for _, b, l in results if b == 1.0) < np.mean([l for _, _, l in results[:8]])
