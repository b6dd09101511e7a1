"""Keras 2.5 Dropout between Dense layers for the oracle fit loop, built on the unchanged pieces of
oracle/keras_mlp.py.  TEST INFRASTRUCTURE ONLY.

[TF-semantics], unpinned like the rest of the oracle: restates tensorflow/python/ops/nn_ops.py ``dropout_v2`` of
TF 2.5 with a number rate, from knowledge of its source:

* ``scale = 1 / (1 - rate)`` (double on the host, rounded to fp32); ``ret = x * scale``; ``ret = ret * cast(keep)``
  with ``keep = random_uniform >= rate``.  Its gradient is Mul's: ``dL/dx = (dL/dret * keep) * scale``; the
  activation's gradient then takes the layer's un-dropped OUTPUT, as TF's activation gradients read the activation
  op's output.
* Keras applies it in training only (``training=True`` inside ``fit``): the epoch loss ``fit`` reports is taken with
  dropout active; ``evaluate`` and ``predict`` see none.

The mask is the project's own (TF's random stream cannot be reproduced), restated here bit for bit: Philox4x32-10
(Random123) with counter (t mod 2^32, t div 2^32, i, 65536 l + j div 4) and key (seed_l, m), word j mod 4, kept when
(w >> 8) 2^-24 >= fp32(rate_l); t is the optimizer state's ``t`` before the step (Keras ``iterations``).

``fit`` reads ``t`` from the state and calls ``km.adam_apply``, ``km._act`` and ``km._act_grad_from_output`` through
the module, so it composes with ``optimizer_oracle.installed()``, ``schedule_oracle.installed()`` and
``activation_oracle.installed()``; a ``regularizer_oracle.Factors`` as ``l2`` adds its l1 terms.
"""
import numpy as np

from oracle import keras_mlp as km
import regularizer_oracle as ro

M0, M1 = 0xD2511F53, 0xCD9E8D57
W0, W1 = 0x9E3779B9, 0xBB67AE85
MASK32 = np.uint64(0xFFFFFFFF)


def philox4x32_10(ctr, key):
    """Philox4x32-10 on uint32 arrays: ctr (4, ...) and key (2, ...) broadcast together; returns (4, ...) uint32.
    The 64-bit products are uint64."""
    c = [np.asarray(x, np.uint64) & MASK32 for x in ctr]
    k0, k1 = (np.asarray(x, np.uint64) & MASK32 for x in key)
    for r in range(10):
        if r:
            k0 = (k0 + np.uint64(W0)) & MASK32
            k1 = (k1 + np.uint64(W1)) & MASK32
        p0 = np.uint64(M0) * c[0]
        p1 = np.uint64(M1) * c[2]
        hi0, lo0 = p0 >> np.uint64(32), p0 & MASK32
        hi1, lo1 = p1 >> np.uint64(32), p1 & MASK32
        c = [hi1 ^ c[1] ^ k0, lo1, hi0 ^ c[3] ^ k1, lo0]
    return np.stack([x.astype(np.uint32) for x in c])


def uniforms(l, t, i, j, seed, m):
    """The uniform u in [0, 1) of hidden layer l, step t, sample positions i, units j, seed, model m (broadcast)."""
    i, j = np.broadcast_arrays(np.asarray(i, np.int64), np.asarray(j, np.int64))
    ctr = (np.full(i.shape, t & 0xFFFFFFFF), np.full(i.shape, t >> 32), i, 65536 * l + (j >> 2))
    w = philox4x32_10(ctr, (np.full(i.shape, seed), np.full(i.shape, m)))
    word = np.take_along_axis(w, (j & 3)[None], 0)[0]
    return (word >> np.uint32(8)).astype(np.float64) * 2.0 ** -24


def keep_mask(l, t, nb, width, rate, seed, m):
    """(nb, width) keep mask of hidden layer l at step t for model m (1.0 kept, 0.0 dropped)."""
    i, j = np.meshgrid(np.arange(nb), np.arange(width), indexing="ij")
    return (uniforms(l, t, i, j, seed, m) >= float(np.float32(rate))).astype(np.float64)


def scale_of(rate):
    return np.float32(1.0 / (1.0 - float(np.float32(rate))))


def loss_and_weight_grads(weights, acts, Xb, zb, masks, rates, l2=0.0, dtype=np.float32, sample_weight=None):
    """The batch loss (mean, or sum(w_i bce_i) / n with sample weights, + penalties) and its gradient with dropout
    masks ``masks[l]`` ((n, width) or None) after hidden layer l."""
    f = dtype
    assert acts[-1] in ("sigmoid", "linear")
    acts_l = list(acts[:-1]) + ["linear"]
    L = len(acts)
    h = np.asarray(Xb).astype(dtype)
    hs, raw = [h], [h]
    for l in range(L):
        a = km._act(acts_l[l], h @ weights[2 * l].astype(dtype, copy=False) + weights[2 * l + 1].astype(dtype))
        raw.append(a)
        if l < L - 1 and masks[l] is not None:
            a = (a * f(scale_of(rates[l]))).astype(dtype) * masks[l].astype(dtype)
        h = a
        hs.append(h)
    u = h
    n = Xb.shape[0]
    z = np.asarray(zb).astype(dtype).reshape(n, 1)
    sw = np.ones((n, 1), dtype) if sample_weight is None else np.asarray(sample_weight).astype(dtype).reshape(n, 1)
    if sample_weight is None:
        loss = f(np.mean(km.bce_with_logits(u, z), dtype=dtype))
        delta = (km._sigmoid(u) - z) / f(n)
    else:
        loss = f(np.sum(sw * km.bce_with_logits(u, z), dtype=dtype) / f(n))
        delta = sw * (km._sigmoid(u) - z) / f(n)
    grads = [None] * len(weights)
    for l in range(L - 1, -1, -1):
        if l < L - 1:
            if masks[l] is not None:  # Mul's gradient, twice: (g keep) scale
                delta = (delta * masks[l].astype(dtype)) * f(scale_of(rates[l]))
            delta = delta * km._act_grad_from_output(acts_l[l], raw[l + 1])
        grads[2 * l] = hs[l].T @ delta
        grads[2 * l + 1] = delta.sum(axis=0)
        if l > 0:
            delta = delta @ weights[2 * l].T
    l2f, l1f = (l2.l2, l2.l1) if isinstance(l2, ro.Factors) else (l2, 0.0)
    l2v = km._l2_vector(l2f, len(weights))
    if any(l2v):
        reg = f(0)
        for i, w in enumerate(weights):
            if l2v[i]:
                reg += f(l2v[i]) * f(np.sum(w * w, dtype=dtype))
                grads[i] = grads[i] + f(2 * l2v[i]) * w
        loss = f(loss + reg)
    return ro._with_l1(loss, grads, weights, l1f, f)


def fit(weights, acts, X, z, epochs, batch_size, permutations, rates, seeds, model=0, state=None, l2=0.0,
        dtype=np.float32, sample_weight=None):
    """km.fit with dropout ``rates[l]`` / ``seeds[l]`` after hidden layer l (rate 0: none) for model index
    ``model``; ``sample_weight`` (N,) per sample.  The masks of a step use ``state.t`` before the update.
    Returns (history (epochs,), state)."""
    X = np.asarray(X).astype(dtype)
    z = np.asarray(z).astype(dtype)
    N = X.shape[0]
    if state is None:
        state = km.AdamState(weights)
    hist = np.zeros(epochs, dtype)
    for e in range(epochs):
        perm = np.asarray(permutations[e])
        tot = dtype(0)
        for s in range(0, N, batch_size):
            idx = perm[s:s + batch_size]
            nb = len(idx)
            masks = [keep_mask(l, int(state.t), nb, weights[2 * l].shape[1], r, sd, model) if r > 0 else None
                     for l, (r, sd) in enumerate(zip(rates, seeds))]
            w = None if sample_weight is None else np.asarray(sample_weight)[idx]
            loss, grads = loss_and_weight_grads(weights, acts, X[idx], z[idx], masks, rates, l2, dtype, w)
            tot += loss * dtype(nb)
            km.adam_apply(weights, grads, state, dtype)
        hist[e] = tot / dtype(N)
    return hist, state
