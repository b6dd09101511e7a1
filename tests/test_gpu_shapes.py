"""The whole net-shape envelope: every kernel against the oracle on nets outside the seven of
helpers.NETS -- one hidden unit, odd widths, the width-128 class, seven hidden layers, D from 1 to
512, no hidden layer -- and at the largest input dimension each (width, depth) accepts.

What takes a net is decided at bore_mlp_create from the kernels' own shared-memory plans
(csrc/mlp_eval.cu, csrc/fit.cu); the CPU tests at the end pin that envelope.  The numbers below
(boundaries, bytes, which fit kernel takes which net and batch, which nets the fused argmax kernel
takes) were derived once from the plan code and are hard-coded, so that a change to a plan shows up
here."""
import ctypes as C
import functools

import numpy as np
import pytest

from oracle import keras_mlp as km, argmax as am
from helpers import trained_weights, synthetic_targets, parallel_minimize_starts

gpu = pytest.mark.gpu

# name: (dims, activations, transform)
SHAPES = {
    "w1": ([3, 1, 1], ["tanh", "sigmoid"], "identity"),                       # one hidden unit
    "odd": ([5, 3, 17, 1], ["elu", "tanh", "sigmoid"], "identity"),           # narrow tiles, uneven U
    "w33": ([7, 33, 1], ["relu", "linear"], "sigmoid"),                       # just past K2's 32-unit mapping
    "w65": ([9, 65, 63, 1], ["relu", "elu", "sigmoid"], "identity"),          # width-128 class, two K2 chunks
    # [12, 128, 128, 1] is refused at create (one-CTA training needs 287,392 B): 128 units once
    "w128": ([12, 128, 64, 1], ["relu", "relu", "sigmoid"], "identity"),
    "w127exp": ([4, 127, 1], ["sigmoid", "linear"], "exp"),                   # exp transform, wide layer
    "deep7": ([6] + [32] * 7 + [1], ["relu"] * 7 + ["sigmoid"], "identity"),  # BORE_MAX_LAYERS
    "deep7_mixed": ([10, 16, 48, 8, 96, 24, 64, 40, 1],
                    ["tanh", "relu", "elu", "sigmoid", "relu", "linear", "elu", "sigmoid"], "identity"),
    "nwn": ([20, 4, 128, 4, 1], ["elu", "tanh", "relu", "sigmoid"], "identity"),  # narrow -> wide -> narrow
    "d1": ([1, 16, 1], ["relu", "sigmoid"], "identity"),
    "d65": ([65, 64, 64, 1], ["relu", "relu", "sigmoid"], "identity"),        # D just past 64
    "d257": ([257, 32, 32, 1], ["tanh", "tanh", "sigmoid"], "identity"),
    # BORE_MAX_DIM: only 16-unit nets train at D = 512 (one-CTA plan); the fused argmax does not fit
    "d512": ([512, 16, 16, 1], ["elu", "elu", "linear"], "sigmoid"),
    "nohid300": ([300, 1], ["sigmoid"], "identity"),
    # the largest D of three (width, depth) pairs; K2 stages 3 / 9 / 9 warps there
    "edge_32x2": ([465, 32, 32, 1], ["tanh", "tanh", "sigmoid"], "identity"),
    "edge_64x3": ([139, 64, 64, 64, 1], ["elu", "elu", "elu", "sigmoid"], "identity"),
    "edge_128x1": ([156, 128, 1], ["tanh", "sigmoid"], "identity"),
}
NAMES = list(SHAPES)
# nets whose fused L-BFGS-B kernel cannot hold weights + two starts in one SM (lbfgsb_fused_fits, m = 10)
NO_FUSED = {"d512", "edge_32x2"}


@functools.lru_cache(maxsize=None)
def _weights(name, seed=1):
    dims, acts, _ = SHAPES[name]
    return tuple(trained_weights(dims, acts, seed=seed, N=200, epochs=10))


def _net(name, n_models=1, seed=1):
    from bore_b200.engine import NativeMLP
    dims, acts, _ = SHAPES[name]
    net = NativeMLP(dims, acts, n_models=n_models)
    net.set_weights(list(_weights(name, seed)))
    return net


# ---------------------------------------------------------------- K0 / K2 against the oracle
RTOL, ATOL = 1e-5, 2e-6  # the bar of test_gpu_mlp_eval.py


@gpu
@pytest.mark.parametrize("S", [1, 17, 1037])
@pytest.mark.parametrize("name", NAMES)
def test_value_grad_and_predict_match_oracle(name, S):
    dims, acts, _ = SHAPES[name]
    w = list(_weights(name))
    net = _net(name)
    X = np.random.RandomState(S + dims[0]).uniform(-0.2, 1.2, size=(S, dims[0]))
    y = net.predict(X)
    y32 = km.predict(w, acts, X)
    assert np.all(np.abs(y - y32) <= RTOL * np.abs(y32) + ATOL), np.abs(y - y32).max()
    for transform in ("identity", "sigmoid", "exp"):
        for negate in (True, False):
            f, g = net.value_and_grad(X, transform, negate)
            f32, g32 = km.value_and_input_grad(w, acts, X, transform, negate, np.float32)
            f64, g64 = km.value_and_input_grad(w, acts, X, transform, negate, np.float64)
            gscale = np.abs(g64).max(axis=1, keepdims=True)
            assert np.all(np.abs(f - f32) <= RTOL * np.abs(f32) + ATOL), (transform, negate, np.abs(f - f32).max())
            assert np.all(np.abs(g - g32) <= RTOL * gscale + ATOL), \
                (transform, negate, (np.abs(g - g32) / (gscale + 1e-30)).max())
            assert np.abs(g - g64).max() <= 4 * np.abs(g32 - g64).max() + ATOL, (transform, negate)


# ---------------------------------------------------------------- fit against the oracle
LOSS_TOL = 1e-4
EPOCHS = 6  # short: long ReLU trajectories separate any two fp32 runs (DESIGN.md section 2)

_UNIT = "unit-split cluster kernel does not take"
_MMA = "tensor-pipe kernel does not take"
# (net, fit mode, batch) -> the error the mode must raise; every other combination must train.
# Mode 4 (K1u) takes no net without a hidden layer, no batch above 64 and no plan above 226 KB; mode 2
# (sample-split cluster) no plan above 226 KB; mode 1 (one CTA) no plan above 227 KB.
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


def _fit_problem(dims, N, epochs, seed):
    rs = np.random.RandomState(seed)
    X = rs.uniform(size=(N, dims[0]))
    y = synthetic_targets(X)
    z = y < np.quantile(y, 0.25)
    perms = np.stack([rs.permutation(N) for _ in range(epochs)])
    return X, z, perms


@functools.lru_cache(maxsize=None)
def _fit_case(name, batch):
    """problem + the oracle's fit of it (shared by the modes)"""
    dims, acts, _ = SHAPES[name]
    N = 40 if batch < 8 else 150  # batch 1: 40 steps per epoch
    X, z, perms = _fit_problem(dims, N, EPOCHS, seed=batch + dims[0])
    w0 = km.init_weights(dims, 3)
    w_ref = [w.copy() for w in w0]
    hist_ref, adam_ref = km.fit(w_ref, acts, X, z, EPOCHS, batch, perms)
    return X, z, perms, w0, hist_ref, w_ref, adam_ref


FIT_CASES = [(n, m, 64) for n in NAMES for m in (1, 2, 4)]
FIT_CASES += [(n, m, b) for n in ("odd", "w65", "deep7_mixed") for m in (1, 2, 4) for b in (1, 5, 100, 128)]
FIT_CASES += [(n, 3, 64) for n in ("odd", "w65", "w128", "deep7_mixed")]


@gpu
@pytest.mark.parametrize("name,mode,batch", FIT_CASES)
def test_fit_matches_oracle(name, mode, batch):
    from bore_b200.engine import NativeMLP
    from bore_b200._lib import BoreNativeError
    dims, acts, _ = SHAPES[name]
    X, z, perms, w0, hist_ref, w_ref, adam_ref = _fit_case(name, batch)
    net = NativeMLP(dims, acts)
    net.set_fit_mode(mode)
    net.set_weights(w0)
    refused = FIT_REFUSED.get((name, mode, batch))
    if refused:
        with pytest.raises(BoreNativeError, match=refused):
            net.fit(X, z, EPOCHS, batch, perms)
        return
    hist = net.fit(X, z, EPOCHS, batch, perms)
    assert np.abs(hist - hist_ref).max() <= LOSS_TOL, np.abs(hist - hist_ref).max()
    for a, b in zip(net.get_weights(), w_ref):
        assert np.abs(a - b).max() <= 2e-3, np.abs(a - b).max()
    m, v, t = net.get_adam_state()
    assert t == adam_ref.t == EPOCHS * (-(-len(X) // batch))
    for a, b in zip(m, adam_ref.m):
        assert np.abs(a - b).max() <= 1e-4
    loss, acc = net.evaluate(X, z)
    loss_ref, acc_ref = km.evaluate(net.get_weights(), acts, X, z)
    assert abs(loss - loss_ref) <= 1e-5 and abs(acc - acc_ref) <= 1e-6


@gpu
@pytest.mark.parametrize("name", ["w65", "deep7_mixed"])
def test_many_models_fit_matches_oracle(name):
    """20 models in one fit_dev call: more than fit the SMs as clusters, so one CTA per model."""
    from bore_b200.engine import NativeMLP
    dims, acts, _ = SHAPES[name]
    M, N, E = 20, 150, EPOCHS
    probs = [_fit_problem(dims, N, E, seed=50 + i) for i in range(M)]
    ws = [km.init_weights(dims, 200 + i) for i in range(M)]
    net = NativeMLP(dims, acts, n_models=M)
    for i, w in enumerate(ws):
        net.set_weights(w, model=i)
    Xd = net.to_device(np.concatenate([p[0] for p in probs]), np.float32)
    zd = net.to_device(np.concatenate([p[1] for p in probs]).astype(np.float32), np.float32)
    pd = net.to_device(np.stack([p[2] for p in probs]).astype(np.int32), np.int32)
    loss = net.fit_dev(Xd, zd, N, 64, E, pd, model0=0, count=M, shared_data=False,
                       shared_perm=False).cpu().numpy()
    for i in range(M):
        w_ref = [w.copy() for w in ws[i]]
        h_ref, _ = km.fit(w_ref, acts, probs[i][0], probs[i][1], E, 64, probs[i][2])
        assert np.abs(loss[i] - h_ref).max() <= LOSS_TOL, (i, np.abs(loss[i] - h_ref).max())
        for u, v in zip(net.get_weights(model=i), w_ref):
            assert np.abs(u - v).max() <= 2e-3


# ---------------------------------------------------------------- argmax: fused kernel vs rounds
KEYS = ("x", "fun", "nit", "nfev", "status", "task")


def _set_lb_mode(mode):
    from bore_b200 import _lib
    _lib.check(_lib.require_cuda().bore_lbfgsb_set_mode(mode))


@pytest.fixture
def lb_mode():
    yield _set_lb_mode
    _set_lb_mode(0)


def _minimize(net, X0, transform, mode):
    import torch
    _set_lb_mode(mode)
    net._work = None
    r = net.lbfgsb_dev(torch.from_numpy(X0).cuda(), 0.0, 1.0, transform=transform)
    return {k: (v.cpu().numpy() if hasattr(v, "cpu") else v) for k, v in r.items()}


@gpu
@pytest.mark.parametrize("name", NAMES)
def test_fused_equals_rounds(name, lb_mode):
    dims, acts, transform = SHAPES[name]
    net = _net(name, seed=5)
    S = 300
    X0 = np.random.RandomState(7).uniform(size=(S, dims[0]))
    _set_lb_mode(0)
    fused_ws = net.lib.bore_lbfgsb_minimize_workspace_bytes(net.h, S, 10)
    rounds_ws = net.lib.bore_lbfgsb_workspace_bytes(S, dims[0], 10)
    b = _minimize(net, X0, transform, 1)
    assert b["rounds"] > 1
    if name in NO_FUSED:
        # the model does not fit beside two starts: the default rule runs rounds, and says so
        assert fused_ws == rounds_ws
        a = _minimize(net, X0, transform, 0)
        assert a["rounds"] == b["rounds"]
    else:
        assert fused_ws < rounds_ws
        a = _minimize(net, X0, transform, 2)
        assert a["rounds"] == 1
    for k in KEYS:
        assert np.array_equal(a[k], b[k]), k
    assert a["evals"] == b["evals"]


@gpu
def test_handover_on_a_width_128_net(lb_mode):
    """n = 20 > 16 and 5,000 starts > 4,096: rounds first, the fused kernel (width-128 class) takes
    the tail over in resume mode -- same results as rounds alone."""
    name = "nwn"
    dims, acts, transform = SHAPES[name]
    net = _net(name, seed=4)
    X0 = np.random.RandomState(11).uniform(size=(5000, dims[0]))
    a = _minimize(net, X0, transform, 0)
    b = _minimize(net, X0, transform, 1)
    assert 1 < a["rounds"] < b["rounds"]
    for k in KEYS:
        assert np.array_equal(a[k], b[k]), k
    assert a["evals"] == b["evals"]


# ---------------------------------------------------------------- argmax against SciPy
# smooth nets on which the reference does not agree with ITSELF on 99 % of these 64 starts after an fp32
# re-association of the MLP (helpers.reference_self_agreement): edge_32x2, 465-D, 0.92 -- local optima
# close in value, reached or missed by an ulp.  They are held to that yardstick, as ReLU nets are.
SELF_AGREEMENT = {"edge_32x2"}


@gpu
@pytest.mark.parametrize("name", NAMES)
def test_minimize_vs_scipy(name):
    from test_gpu_lbfgsb import FUN_TOL, _check_against_self_agreement
    dims, acts, transform = SHAPES[name]
    n = dims[0]
    w = list(_weights(name, seed=7))
    net = _net(name, seed=7)
    X0 = np.random.RandomState(11).uniform(size=(64, n))
    got = net.lbfgsb(X0, 0.0, 1.0, transform=transform)
    ref = parallel_minimize_starts(w, acts, X0, 0.0, 1.0, transform)
    agree = np.abs(got["fun"] - ref["fun"]) <= FUN_TOL
    print(name, "agree", agree.mean(), "rounds", got["rounds"])
    if "relu" in acts or name in SELF_AGREEMENT:
        _check_against_self_agreement(name, got, ref, w, acts, transform, X0, n)
    else:
        assert agree.mean() >= 0.99, agree.mean()
    assert np.all(got["x"] >= 0.0) and np.all(got["x"] <= 1.0)
    f_chk, _ = km.value_and_input_grad(w, acts, got["x"], transform, True, np.float32)
    assert np.abs(f_chk - got["fun"]).max() <= 1e-5
    assert set(np.unique(got["status"])) <= {0, 1, 2}


# ---------------------------------------------------------------- batched problems
@gpu
@pytest.mark.parametrize("name", ["w128", "deep7_mixed", "d257"])
def test_batched_problems(name, lb_mode):
    import torch
    dims, acts, transform = SHAPES[name]
    M, P, K = 5, 40, 8
    net = _net(name, n_models=M)
    for p in range(1, M):
        net.set_weights(list(_weights(name, seed=20 + p)), model=p)
    Xq = np.random.RandomState(3).uniform(size=(M, P, dims[0]))
    multi = net.predict_multi_dev(torch.from_numpy(Xq.astype(np.float32)).cuda()).cpu().numpy()
    for p in range(M):
        assert np.array_equal(multi[p], net.predict(Xq[p], model=p)[:, 0]), p
    X0 = np.random.RandomState(5).uniform(size=(M, K, dims[0]))
    out = []
    for mode in (2, 1):
        _set_lb_mode(mode)
        net._work = None
        r = net.lbfgsb_multi_dev(torch.from_numpy(X0).cuda(), 0.0, 1.0, transform=transform)
        out.append({k: (v.cpu().numpy() if hasattr(v, "cpu") else v) for k, v in r.items()})
    for k in KEYS:
        assert np.array_equal(out[0][k], out[1][k]), k


# ---------------------------------------------------------------- the envelope at create (no GPU needed)
_LIMIT = "(limit 232448 B)"  # 227 KB of shared memory per CTA


def _create(dims):
    """bore_mlp_create's verdict on a net: None when it was created, else the error text."""
    from bore_b200 import _lib
    from bore_b200.engine import ACT_CODES
    lib = _lib.load()
    acts = ["tanh"] * (len(dims) - 2) + ["sigmoid"]
    h = C.c_void_p()
    rc = lib.bore_mlp_create(len(acts), (C.c_int * len(dims))(*dims),
                             (C.c_int * len(acts))(*[ACT_CODES[a] for a in acts]), 1, 0, C.byref(h))
    if rc == 0:
        lib.bore_mlp_destroy(h)
        return None
    return lib.bore_last_error().decode()


def _assert_accepted(dims):
    from bore_b200 import _lib
    err = _create(dims)
    if _lib.load().bore_device_count() > 0:
        assert err is None, (dims, err)
    else:  # the envelope check passed and the device check is what refused it
        assert err == "bore_mlp_create: no CUDA device visible -- bore_b200 has no CPU fallback", (dims, err)


# (hidden widths, largest accepted D, what D + 1 needs): one-CTA training at batch 64 is the binding
# plan at every boundary
EDGES = [
    ([32, 32], 465, 232848),
    ([64, 64, 64], 139, 232608),
    ([128], 156, 232624),
    ([65, 65], 224, 232880),
    ([32] * 7, 245, 232528),
]


@pytest.mark.parametrize("hidden,dmax,need", EDGES)
def test_create_accepts_up_to_the_largest_input_dim(hidden, dmax, need):
    _assert_accepted([dmax] + hidden + [1])
    err = _create([dmax + 1] + hidden + [1])
    assert err == f"bore_mlp_create: training at batch 64 needs {need} B of shared memory per model {_LIMIT}", err


@pytest.mark.parametrize("dims", [v[0] for v in SHAPES.values()] +
                         [[512] + [16] * 7 + [1], [512, 1], [1, 128, 1], [1] + [2] * 7 + [1]])
def test_create_accepts_the_test_nets(dims):
    _assert_accepted(dims)


@pytest.mark.parametrize("dims,what", [
    ([8, 128, 128, 128, 128, 1], "predict (K0) needs 234752 B of shared memory for one warp"),
    ([300, 128, 128, 1], "predict (K0) needs 254464 B of shared memory for one warp"),
    ([129, 128, 128, 128, 1], "value and gradient (K2) needs 263616 B of shared memory for one warp"),
    ([12, 128, 128, 1], "training at batch 64 needs 287392 B of shared memory per model"),
    ([512, 64, 64, 1], "training at batch 64 needs 377568 B of shared memory per model"),
    ([512, 32, 1], "training at batch 64 needs 233712 B of shared memory per model"),
])
def test_create_refuses_nets_no_kernel_can_run(dims, what):
    assert _create(dims) == f"bore_mlp_create: {what} {_LIMIT}"
