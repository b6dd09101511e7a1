"""Ragged batched problems on the GPU: problems of one launch with their own observation counts N_p and
epochs (bore_mlp_fit_ragged), their own quantile labels (bore_quantile_labels_ragged) and their own stored
rows for the duplicate filter (bore_is_duplicate_ragged).  Per problem the result must be the
single-problem fit / argmax: bit for bit against the uniform launch and a lone launch where the plan is
the same, against the oracle otherwise."""
import numpy as np
import pytest

from oracle import keras_mlp as km, argmax as am
import weighted_oracle as wo
from helpers import NETS, synthetic_targets

pytestmark = pytest.mark.gpu

SHAPES = {n: (d, list(a)) for n, (d, a, _) in NETS.items()}
SHAPES["odd"] = ([5, 3, 17, 1], ["elu", "tanh", "sigmoid"])  # the run-time-shape K1u build
SHAPES["w65"] = ([9, 65, 63, 1], ["relu", "elu", "sigmoid"])
LOSS_TOL = 1e-4

# the mixed sizes: every N_p with two different epoch counts
N_SET = (1, 7, 63, 64, 65, 150, 500, 1037)
E_SET = (0, 1, 3, 8)
MIX_N = [N_SET[i % 8] for i in range(16)]
MIX_E = [E_SET[(i + i // 8) % 4] for i in range(16)]


def _problem(D, N, E, seed):
    rs = np.random.RandomState(seed)
    X = rs.uniform(size=(N, D))
    y = synthetic_targets(X) + 0.1 * seed * X[:, 0]
    z = y < np.quantile(y, 0.3)
    perms = np.array([rs.permutation(N) for _ in range(E)], dtype=np.int64).reshape(E, N)
    w = rs.uniform(0.0, 2.0, size=N).astype(np.float32)
    return X, z, perms, w


def _problems(D, ns, es, seed=0):
    return [_problem(D, n, e, seed + 7 * p) for p, (n, e) in enumerate(zip(ns, es))]


def _net(dims, acts, mode, ws):
    from bore_b200.engine import NativeMLP
    net = NativeMLP(dims, acts, n_models=len(ws))
    net.set_fit_mode(mode)
    for i, w in enumerate(ws):
        net.set_weights(w, model=i)
    return net


def _ragged(net, probs, es, batch, weighted, cw=None):
    """One bore_mlp_fit_ragged launch over `probs` -> (M, max epochs) losses (NaN padded)."""
    from bore_b200.ragged import RaggedLayout
    lay = RaggedLayout([len(p[0]) for p in probs], es)
    X = np.concatenate([p[0] for p in probs])
    z = np.concatenate([p[1] for p in probs]).astype(np.float32)
    perm = np.concatenate([p[2].reshape(-1) for p in probs]).astype(np.int32)
    w = net.to_device(np.concatenate([p[3] for p in probs]), np.float32) if weighted else None
    loss = net.fit_ragged_dev(net.to_device(X, np.float32), net.to_device(z, np.float32), lay, batch,
                              net.to_device(perm, np.int32), w_dev=w, class_weight=cw)
    return lay.pad_loss(loss.cpu().numpy())


def _state(net, i):
    m, v, t = net.get_adam_state(model=i)
    return net.get_weights(model=i), m, v, t


def _assert_same_state(a, b, what):
    wa, ma, va, ta = a
    wb, mb, vb, tb = b
    assert ta == tb, what
    for x, y in zip(wa + ma + va, wb + mb + vb):
        assert np.array_equal(x, y), what


def _assert_same_loss(a, b, what):
    assert np.array_equal(np.isnan(a), np.isnan(b)) and np.array_equal(a[~np.isnan(a)], b[~np.isnan(b)]), what


# ---------------------------------------------------------------- 1. equal N_p: the uniform launch, bit for bit
CASES1 = [(n, m, 6, wt) for n in ("cfg3_ackley50", "odd") for m in (1, 2, 3, 4) for wt in (False, True)]
CASES1 += [("cfg2_hartmann6", 1, 600, wt) for wt in (False, True)]


@pytest.mark.parametrize("name,mode,M,weighted", CASES1)
def test_equal_counts_are_the_uniform_launch_bit_for_bit(name, mode, M, weighted):
    from bore_b200._lib import BoreNativeError
    dims, acts = SHAPES[name]
    N, E, B = 150, 4, 64
    probs = _problems(dims[0], [N] * M, [E] * M, seed=1)
    ws = [km.init_weights(dims, 30 + i % 50) for i in range(M)]
    cw = (0.5, 2.0) if weighted else None
    uni = _net(dims, acts, mode, ws)
    X = np.concatenate([p[0] for p in probs])
    z = np.concatenate([p[1] for p in probs]).astype(np.float32)
    perm = np.stack([p[2] for p in probs]).astype(np.int32)
    w = uni.to_device(np.concatenate([p[3] for p in probs]), np.float32) if weighted else None
    try:
        loss_u = uni.fit_dev(uni.to_device(X, np.float32), uni.to_device(z, np.float32), N, B, E,
                             uni.to_device(perm, np.int32), model0=0, count=M, shared_data=False,
                             shared_perm=False, w_dev=w, class_weight=cw).cpu().numpy()
        error = None
    except BoreNativeError as e:
        error = str(e)
    rag = _net(dims, acts, mode, ws)
    if error is not None:  # refused: with the same words
        with pytest.raises(BoreNativeError) as info:
            _ragged(rag, probs, [E] * M, B, weighted, cw)
        assert str(info.value) == error
        return
    loss_r = _ragged(rag, probs, [E] * M, B, weighted, cw)
    assert np.array_equal(loss_u, loss_r)
    for i in list(range(min(M, 6))) + [M - 1]:
        _assert_same_state(_state(uni, i), _state(rag, i), i)


# ---------------------------------------------------------------- 2. mixed sizes against the oracle
CASES2 = [("cfg2_hartmann6", m, 64) for m in (1, 2, 3, 4)]
CASES2 += [(n, m, b) for n in ("odd", "w65", "cfg5_plugin8") for m in (1, 2) for b in (5, 128)]


@pytest.mark.parametrize("weighted", [False, True])
@pytest.mark.parametrize("name,mode,batch", CASES2)
def test_mixed_sizes_match_the_oracle_per_problem(name, mode, batch, weighted):
    dims, acts = SHAPES[name]
    probs = _problems(dims[0], MIX_N, MIX_E, seed=2)
    ws = [km.init_weights(dims, 60 + i) for i in range(len(probs))]
    cw = (0.7, 1.6) if weighted else None
    net = _net(dims, acts, mode, ws)
    hist = _ragged(net, probs, MIX_E, batch, weighted, cw)
    assert hist.shape == (len(probs), max(MIX_E))
    for i, (X, z, perms, w) in enumerate(probs):
        E = MIX_E[i]
        w_ref = [a.copy() for a in ws[i]]
        kw = dict(sample_weight=w, class_weight={0: cw[0], 1: cw[1]}) if weighted else {}
        h_ref, adam = wo.fit(w_ref, acts, X, z, E, batch, perms, **kw)
        assert np.isnan(hist[i, E:]).all(), i
        if E:
            assert np.abs(hist[i, :E] - h_ref).max() <= LOSS_TOL, (i, np.abs(hist[i, :E] - h_ref).max())
        got_w, m, v, t = _state(net, i)
        assert t == adam.t == E * (-(-len(X) // batch)), i
        for a, b in zip(got_w, w_ref):
            assert np.abs(a - b).max() <= 2e-3, (i, np.abs(a - b).max())
        for a, b in zip(m, adam.m):
            assert np.abs(a - b).max() <= 1e-4, i


# ---------------------------------------------------------------- 3. a problem alone gives the same bits
@pytest.mark.parametrize("mode", [0, 1, 2, 3, 4])
def test_problems_with_a_full_batch_are_their_lone_launch_bit_for_bit(mode):
    dims, acts = SHAPES["cfg2_hartmann6"]
    B = 64
    probs = _problems(dims[0], MIX_N, MIX_E, seed=3)
    ws = [km.init_weights(dims, 90 + i) for i in range(len(probs))]
    net = _net(dims, acts, mode, ws)
    hist = _ragged(net, probs, MIX_E, B, True, (0.8, 1.3))
    checked = 0
    for i, (X, z, perms, w) in enumerate(probs):
        if len(X) < B or MIX_E[i] == 0:
            continue
        lone = _net(dims, acts, mode, [ws[i]])
        h = lone.fit(X, z, MIX_E[i], B, perms, w=w, class_weight=(0.8, 1.3))
        assert np.array_equal(h, hist[i, :MIX_E[i]]), i
        _assert_same_state(_state(lone, 0), _state(net, i), i)
        checked += 1
    assert checked >= 6


# ---------------------------------------------------------------- 4. epochs_p = 0, and the problem order
@pytest.mark.parametrize("mode", [0, 1])
def test_zero_epochs_leave_a_problem_untouched_and_order_does_not_matter(mode):
    dims, acts = SHAPES["cfg5_plugin8"]
    M = len(MIX_N)
    probs = _problems(dims[0], MIX_N, [2] * M, seed=4)
    ws = [km.init_weights(dims, 120 + i) for i in range(M)]
    net = _net(dims, acts, mode, ws)
    _ragged(net, probs, [2] * M, 32, False)  # non-trivial weights and Adam state everywhere
    before = [_state(net, i) for i in range(M)]
    probs = _problems(dims[0], MIX_N, MIX_E, seed=5)
    hist = _ragged(net, probs, MIX_E, 32, False)
    after = [_state(net, i) for i in range(M)]
    for i in range(M):
        if MIX_E[i] == 0:
            _assert_same_state(before[i], after[i], i)
            assert np.isnan(hist[i]).all()
        else:
            assert after[i][3] > before[i][3]
    # the same problems in the reverse order (model M-1-i holds problem i): the same bits per problem
    rev = _net(dims, acts, mode, [ws[M - 1 - i] for i in range(M)])
    _ragged(rev, _problems(dims[0], MIX_N, [2] * M, seed=4)[::-1], [2] * M, 32, False)
    hist_r = _ragged(rev, probs[::-1], MIX_E[::-1], 32, False)
    for i in range(M):
        _assert_same_state(after[i], _state(rev, M - 1 - i), i)
        _assert_same_loss(hist[i], hist_r[M - 1 - i], i)


def test_nothing_to_train_is_a_no_op():
    dims, acts = SHAPES["cfg2_hartmann6"]
    probs = _problems(dims[0], [5, 9], [0, 0], seed=6)
    ws = [km.init_weights(dims, 7), km.init_weights(dims, 8)]
    net = _net(dims, acts, 0, ws)
    hist = _ragged(net, probs, [0, 0], 64, False)
    assert hist.shape == (2, 0)
    for i in range(2):
        w, m, v, t = _state(net, i)
        assert t == 0 and all(np.array_equal(a, b) for a, b in zip(w, ws[i]))


# ---------------------------------------------------------------- 5. per-budget-like problems: one cluster each
def test_few_problems_run_one_cluster_each():
    dims, acts = SHAPES["cfg5_plugin8"]
    ns, es = [27, 81, 243], [12, 6, 3]
    probs = _problems(dims[0], ns, es, seed=7)
    ws = [km.init_weights(dims, 150 + i) for i in range(3)]
    got = {}
    for mode in (4, 0):
        net = _net(dims, acts, mode, ws)
        got[mode] = (_ragged(net, probs, es, 64, True, (1.0, 3.0)), [_state(net, i) for i in range(3)])
    for i in range(3):  # automatic mode picks the unit-split cluster kernel for three problems
        _assert_same_state(got[4][1][i], got[0][1][i], i)
        _assert_same_loss(got[4][0][i], got[0][0][i], i)
    for i, (X, z, perms, w) in enumerate(probs):
        w_ref = [a.copy() for a in ws[i]]
        h_ref, adam = wo.fit(w_ref, acts, X, z, es[i], 64, perms, sample_weight=w, class_weight={0: 1.0, 1: 3.0})
        assert np.abs(got[4][0][i, :es[i]] - h_ref).max() <= LOSS_TOL, i
        assert got[4][1][i][3] == adam.t
        for a, b in zip(got[4][1][i][0], w_ref):
            assert np.abs(a - b).max() <= 2e-3, i
        # the compile-time K1u build pads every batch to 64 samples: a lone launch has the same plan
        lone = _net(dims, acts, 4, [ws[i]])
        h = lone.fit(X, z, es[i], 64, perms, w=w, class_weight=(1.0, 3.0))
        assert np.array_equal(h, got[4][0][i, :es[i]]), i
        _assert_same_state(_state(lone, 0), got[4][1][i], i)


# ---------------------------------------------------------------- 6. ragged quantile labels
def test_ragged_quantile_labels_are_numpys():
    from bore_b200.engine import NativeMLP
    from bore_b200._lib import BoreNativeError
    net = NativeMLP([2, 4, 1], ["relu", "sigmoid"])
    rs = np.random.RandomState(8)
    ns = [1, 2, 3, 17, 100, 1000, 16384, 5, 64, 777]
    ys = [rs.normal(size=n) for n in ns]
    ys[3][4] = np.nan                  # a problem holding NaN: tau NaN, no positives
    ys[4][::3] = ys[4][1]              # ties
    ys[8][:] = 0.5                     # constant
    ys[9][:10] = -0.0
    for gamma in (0.25, 1 / 3, 0.0, 1.0):
        z, tau = net.quantile_labels_ragged_dev(net.to_device(np.concatenate(ys), np.float64), ns, gamma,
                                                want_tau=True)
        z, tau = z.cpu().numpy(), tau.cpu().numpy()
        off = np.concatenate([[0], np.cumsum(ns)])
        for p, y in enumerate(ys):
            t = np.quantile(y, gamma)
            assert np.array_equal(tau[p], t, equal_nan=True), (gamma, p)
            assert np.array_equal(z[off[p]:off[p + 1]], np.less(y, t).astype(np.float32)), (gamma, p)
    with pytest.raises(BoreNativeError, match="exceeds the shared-memory sort"):
        net.quantile_labels_ragged_dev(net.to_device(np.zeros(16385 + 3), np.float64), [3, 16385], 0.25)


# ---------------------------------------------------------------- 7. ragged duplicate filter
def test_ragged_duplicate_filter_is_record_is_duplicate():
    from bore_b200.data import Record
    from bore_b200.engine import NativeMLP
    net = NativeMLP([3, 4, 1], ["relu", "sigmoid"])
    rs = np.random.RandomState(9)
    G, K, D = 6, 40, 3
    n_prev = [0, 1, 5, 37, 0, 200]
    prev = [rs.uniform(size=(n, D)) for n in n_prev]
    x = rs.uniform(size=(G, K, D))
    for g in range(G):  # exact and near copies of stored rows, and copies of another group's rows
        if n_prev[g]:
            x[g, :10] = prev[g][rs.randint(n_prev[g], size=10)]
            x[g, 10:15] = x[g, 10:15] * 0 + prev[g][0] * (1 + 1e-7)
            x[g, 15:18] = prev[g][0] + 1e-3
        x[g, 18:20] = prev[5][:2]
    keep = net.keep_unique_ragged_dev(net.to_device(x, np.float64), n_prev,
                                      net.to_device(np.concatenate(prev), np.float64)).cpu().numpy()
    for g in range(G):
        rec = Record()
        for r in prev[g]:
            rec.append(r, 0.0)
        for c in range(K):
            assert keep[g, c] == (0 if rec.is_duplicate(x[g, c]) else 1), (g, c)
    assert keep[0].all() and keep[4].all() and not keep[5, :15].any() and not keep[5, 18:20].any()


# ---------------------------------------------------------------- 8. end to end through the batched surface
def test_ragged_fit_and_argmax_match_the_oracle_per_problem():
    from scipy.optimize import Bounds
    from bore_b200 import BatchedMaximizableSequential, Dense, BinaryCrossentropy, sigmoid
    D, gamma, cw = 6, 1 / 3, {0: 0.8, 1: 2.5}
    ns, es = [150, 23, 64, 400, 9, 97], [8, 3, 0, 2, 20, 5]
    M = len(ns)
    dims, acts = [D, 32, 32, 32, 1], ["elu", "elu", "elu", "linear"]  # the plugin's network
    rs = np.random.RandomState(10)
    X = [rs.uniform(size=(n, D)) for n in ns]
    y = [synthetic_targets(X[p]) + 0.3 * p * X[p][:, 0] for p in range(M)]
    sw = [rs.uniform(0.2, 2.0, size=n) for n in ns]
    layers = [Dense(32, activation="elu", input_dim=D), Dense(32, activation="elu"),
              Dense(32, activation="elu"), Dense(1)]
    model = BatchedMaximizableSequential(layers, n_problems=M, transform=sigmoid, seed=1)
    model.compile(optimizer="adam", loss=BinaryCrossentropy(from_logits=True))
    w0 = [km.init_weights(dims, 10 + p) for p in range(M)]
    model.set_weights(w0)
    # the surface draws the permutations from the model's generator: problem after problem, epoch after epoch
    draw = np.random.RandomState(1)
    for p in range(M):  # (what the constructor's glorot draws consumed)
        for fi, fo in zip(dims[:-1], dims[1:]):
            draw.uniform(size=(fi, fo))
    perms = [np.array([draw.permutation(ns[p]) for _ in range(es[p])], dtype=np.int64).reshape(es[p], ns[p])
             for p in range(M)]
    hist = model.fit(X, y, batch_size=64, epochs=es, gamma=gamma, sample_weight=sw, class_weight=cw, verbose=1)
    assert hist.shape == (M, max(es)) and hist.epochs.tolist() == es
    got_w = model.get_weights()
    for p in range(M):
        z = y[p] < np.quantile(y[p], gamma)
        w = [a.copy() for a in w0[p]]
        h_ref, _ = wo.fit(w, acts, X[p], z, es[p], 64, perms[p], sample_weight=sw[p], class_weight=cw)
        assert np.abs(hist[p, :es[p]] - h_ref).max(initial=0) <= LOSS_TOL, p
        assert np.isnan(hist[p, es[p]:]).all()
        for a, b in zip(got_w[p], w):
            np.testing.assert_allclose(a, b, rtol=2e-4, atol=2e-4)

    bounds = Bounds(np.zeros(D), np.ones(D))
    res0 = model.argmax(bounds, num_starts=4, num_samples=128, random_state=np.random.RandomState(5))
    # exclude: problem 1 stores its own winner (so it must be filtered), problem 2 stores nothing
    exclude = [X[p] for p in range(M)]
    exclude[1] = np.vstack([X[1], res0[1].x[None]]) if res0[1] is not None else X[1]
    exclude[2] = np.zeros((0, D))
    res = model.argmax(bounds, num_starts=4, num_samples=128, random_state=np.random.RandomState(5),
                       exclude=exclude)
    rs = np.random.RandomState(5)
    from bore_b200.data import Record
    for p in range(M):
        rec = Record()
        for r in exclude[p]:
            rec.append(r, 0.0)
        ref = am.argmax(got_w[p], acts, bounds, filter_fn=lambda r: not rec.is_duplicate(r.x), num_starts=4,
                        num_samples=128, print_fn=lambda s: None, random_state=rs, transform="sigmoid")
        assert (res[p] is None) == (ref is None), p
        if ref is not None:
            assert abs(float(res[p].fun) - float(ref.fun)) <= 1e-4, (p, res[p].fun, ref.fun)
            assert not rec.is_duplicate(res[p].x)
    with pytest.raises(ValueError):
        model.fit(X, y[:-1], epochs=1)
    with pytest.raises(ValueError):
        model.fit(X, y, epochs=[1] * (M + 1))
    with pytest.raises(ValueError):
        model.argmax(bounds, num_starts=4, num_samples=128, random_state=0, exclude=exclude[:-1])
