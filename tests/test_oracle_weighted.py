"""The weighted oracle (tests/weighted_oracle.py: Keras ``sample_weight`` / ``class_weight``) against an
independent torch implementation in fp64, the class-weight rules, and the host-side checks of the
model surface.  CPU only."""
import os

import numpy as np
import pytest
import torch

from oracle import keras_mlp as km
import weighted_oracle as wo
from helpers import NETS

GOLD = os.path.join(os.path.dirname(__file__), "golden")
F = torch.nn.functional
ACT = {"linear": lambda t: t, "relu": torch.relu, "elu": F.elu, "sigmoid": torch.sigmoid, "tanh": torch.tanh}


def _fit_acts(name):
    dims, acts, _ = NETS[name]
    return dims, list(acts[:-1]) + ["sigmoid" if acts[-1] == "sigmoid" else "linear"]


def _torch_loss(ws, acts, X, z, w, l2):
    """torch's own BCE-with-logits with per-element weights; reduction="mean" divides by the
    element count, which is Keras' SUM_OVER_BATCH_SIZE."""
    h = X
    for l, a in enumerate(acts):
        h = h @ ws[2 * l] + ws[2 * l + 1]
        if l < len(acts) - 1:
            h = ACT[a](h)
    loss = F.binary_cross_entropy_with_logits(h, z, weight=w, reduction="mean")
    if l2:
        loss = loss + sum(l2 * (a * a).sum() for a in ws)
    return loss


def _torch_weighted_fit(w0, acts, X, z, sw, epochs, batch, perms, l2=0.0, lr=1e-3, b1=0.9, b2=0.999, eps=1e-7):
    """The pattern of test_oracle._torch_fit (autograd, textbook Adam) with per-sample weights."""
    ws = [torch.tensor(np.asarray(a, np.float64), requires_grad=True) for a in w0]
    m = [torch.zeros_like(a) for a in ws]
    v = [torch.zeros_like(a) for a in ws]
    Xt = torch.tensor(np.asarray(X, np.float64))
    zt = torch.tensor(np.asarray(z, np.float64)).reshape(-1, 1)
    wt = torch.tensor(np.asarray(sw, np.float64)).reshape(-1, 1)
    N, t, hist = Xt.shape[0], 0, []
    for e in range(epochs):
        tot = 0.0
        perm = torch.as_tensor(np.asarray(perms[e], np.int64))
        for s in range(0, N, batch):
            idx = perm[s:s + batch]
            loss = _torch_loss(ws, acts, Xt[idx], zt[idx], wt[idx], l2)
            grads = torch.autograd.grad(loss, ws)
            tot += float(loss.detach()) * len(idx)
            t += 1
            lr_t = lr * np.sqrt(1.0 - b2 ** t) / (1.0 - b1 ** t)
            with torch.no_grad():
                for i, g in enumerate(grads):
                    m[i] = b1 * m[i] + (1.0 - b1) * g
                    v[i] = b2 * v[i] + (1.0 - b2) * g * g
                    ws[i] -= lr_t * m[i] / (torch.sqrt(v[i]) + eps)
        hist.append(tot / N)
    return np.array(hist), [a.detach().numpy() for a in ws], t


def _problem(dims, N, seed):
    rs = np.random.RandomState(seed)
    X = rs.uniform(size=(N, dims[0]))
    y = np.sum((X - 0.45) ** 2, axis=1)
    z = y < np.quantile(y, 0.3)
    w = rs.uniform(0.0, 3.0, size=N)
    w[rs.uniform(size=N) < 0.2] = 0.0
    return rs, X, z, w


@pytest.mark.parametrize("name,l2", [("cfg2_hartmann6", 0.0), ("cfg5_plugin8", 1e-4), ("tanh_exp", 0.0),
                                     ("cfg1_branin", 1e-3)])
def test_weighted_loss_and_grads_vs_torch(name, l2):
    dims, acts = _fit_acts(name)
    _, X, z, w = _problem(dims, 50, 1)
    w0 = km.init_weights(dims, 4, np.float64)
    loss, grads = wo.loss_and_weight_grads(w0, acts, X, z, l2, np.float64, sample_weight=w)
    ws = [torch.tensor(a, dtype=torch.float64, requires_grad=True) for a in w0]
    lt = _torch_loss(ws, acts, torch.tensor(X), torch.tensor(z, dtype=torch.float64).reshape(-1, 1),
                     torch.tensor(w).reshape(-1, 1), l2)
    lt.backward()
    assert abs(loss - lt.item()) <= 1e-12
    for g, p in zip(grads, ws):
        assert np.allclose(g, p.grad.numpy(), rtol=1e-9, atol=1e-12)


@pytest.mark.parametrize("name,l2", [("cfg2_hartmann6", 0.0), ("cfg5_plugin8", 1e-4), ("tanh_exp", 0.0),
                                     ("cfg1_branin", 0.0)])
def test_weighted_fit_vs_torch(name, l2):
    """100 fp64 steps (the last batch of each epoch short) with sample AND class weights."""
    dims, acts = _fit_acts(name)
    rs, X, z, w = _problem(dims, 150, 12)
    E, B = 34, 64
    perms = np.stack([rs.permutation(150) for _ in range(E)])
    cw = {0: 0.5, 1: 2.5}
    w0 = km.init_weights(dims, 3, np.float64)
    wk = [a.copy() for a in w0]
    hist, adam = wo.fit(wk, acts, X, z, E, B, perms, l2=l2, dtype=np.float64, sample_weight=w, class_weight=cw)
    eff = w * np.where(z, 2.5, 0.5)
    hist_t, w_t, t = _torch_weighted_fit(w0, acts, X, z, eff, E, B, perms, l2=l2)
    assert adam.t == t == 102
    assert np.abs(hist - hist_t).max() <= 1e-10, np.abs(hist - hist_t).max()
    assert max(np.abs(a - b).max() for a, b in zip(wk, w_t)) <= 1e-10


def test_unit_weights_are_the_unweighted_oracle_and_the_golden():
    g = np.load(os.path.join(GOLD, "fit_golden.npz"))
    for name in ("cfg1_branin", "cfg5_plugin8"):
        dims, acts, _ = NETS[name]
        w, o = [], 0
        flat = g[name + "/w0"]
        for fi, fo in zip(dims[:-1], dims[1:]):
            w.append(flat[o:o + fi * fo].reshape(fi, fo).copy()); o += fi * fo
            w.append(flat[o:o + fo].copy()); o += fo
        perms, X, z, l2 = g[name + "/perms"], g[name + "/X"], g[name + "/z"], float(g[name + "/l2"])
        runs = {}
        for key, fit, kw in (("none", km.fit, {}),
                             ("ones", wo.fit, dict(sample_weight=np.ones(len(X)), class_weight={0: 1, 1: 1}))):
            wk = [a.copy() for a in w]
            runs[key] = fit(wk, acts, X, z, len(perms), 64, perms, l2=l2, **kw)[0], wk
        assert np.abs(runs["none"][0] - g[name + "/loss"]).max() <= 1e-5
        assert np.array_equal(runs["none"][0], runs["ones"][0])
        for a, b in zip(runs["none"][1], runs["ones"][1]):
            assert np.array_equal(a, b)


# ---------------------------------------------------------------------------- class_weight rules
def test_class_weight_multiplies_sample_weight():
    z = np.array([0, 1, 1, 0, 1], np.float32)
    sw = np.array([1.0, 2.0, 0.0, -1.0, 0.5])
    assert np.allclose(wo.sample_weights(z, sw, {0: 3.0, 1: 0.5}), [3.0, 1.0, 0.0, -3.0, 0.25])
    assert np.allclose(wo.sample_weights(z, None, {0: 3.0, 1: 0.5}), [3.0, 0.5, 0.5, 3.0, 0.5])
    assert np.allclose(wo.sample_weights(z, sw[:, None]), sw)
    assert wo.sample_weights(z) is None
    # more classes than labels use: fine (Keras gathers only the classes present)
    assert np.allclose(wo.sample_weights(z, None, {0: 1.0, 1: 2.0, 2: 7.0}), [1, 2, 2, 1, 2])


@pytest.mark.parametrize("cw", [{1: 1.0, 2: 1.0}, {0: 1.0, 2: 1.0}, {"0": 1.0, "1": 1.0}])
def test_class_weight_keys_must_be_0_to_k(cw):
    from bore_b200.models import sample_weights
    z = np.array([0, 1, 0], np.float32)
    with pytest.raises((ValueError, TypeError)):
        wo.sample_weights(z, None, cw)
    with pytest.raises((ValueError, TypeError)):
        sample_weights(z, None, cw)


def test_label_without_class_weight_key_and_bad_shapes_refused():
    from bore_b200.models import sample_weights
    z = np.array([0, 1, 0], np.float32)
    for fn in (wo.sample_weights, sample_weights):
        with pytest.raises(ValueError):
            fn(z, None, {0: 2.0})
        for bad in (np.ones(4), np.ones((3, 2)), np.ones((1, 3)), np.ones(())):
            with pytest.raises(ValueError):
                fn(z, bad)


def test_model_surface_weights_match_the_oracle_rule():
    from bore_b200.models import sample_weights
    rs = np.random.RandomState(0)
    z = rs.uniform(size=40) < 0.3
    sw = rs.normal(size=(40, 1))
    cw = {0: 0.25, 1: 4.0}
    assert np.array_equal(sample_weights(z, sw, cw), wo.sample_weights(z, sw, cw))


def test_weighted_evaluate_rules():
    dims, acts = _fit_acts("cfg2_hartmann6")
    _, X, z, w = _problem(dims, 60, 3)
    wts = km.init_weights(dims, 5, np.float64)
    loss, acc = wo.evaluate(wts, acts, X, z, dtype=np.float64, sample_weight=w)
    u = km.forward(wts, list(acts[:-1]) + ["linear"], X, np.float64)[:, 0]
    out = km.forward(wts, acts, X, np.float64)[:, 0]
    hit = (out > 0.5) == z
    assert abs(loss - np.sum(w * km.bce_with_logits(u, z)) / 60) <= 1e-12
    assert abs(acc - np.sum(w * hit) / np.sum(w)) <= 1e-12
    # all weights zero: loss 0, accuracy 0 (div_no_nan)
    assert wo.evaluate(wts, acts, X, z, dtype=np.float64, sample_weight=np.zeros(60)) == [0.0, 0.0]
    # unit weights: the unweighted result (the fp32 accuracy is a float32 sum over a sum of ones)
    assert np.allclose(wo.evaluate(wts, acts, X, z, sample_weight=np.ones(60)), km.evaluate(wts, acts, X, z),
                       rtol=0, atol=1e-7)
