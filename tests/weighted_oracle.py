"""Keras' weighted training rules (``sample_weight`` / ``class_weight``) in NumPy, on top of the
oracle's unweighted restatement (oracle/keras_mlp.py: forward pass, BCE-with-logits, activation
gradients, Adam).  TEST INFRASTRUCTURE ONLY.  [TF-semantics], unpinned like the rest of the Keras
half of the oracle; tests/test_oracle_weighted.py checks it against an independent torch
implementation in fp64.

The TF 2.5 sources each rule restates (paths inside the tensorflow repository at tag v2.5.0; cited
from knowledge of that tree):

* sample weights        keras/utils/losses_utils.py ``compute_weighted_loss``: losses * sample_weight,
                        then SUM_OVER_BATCH_SIZE = sum / number of samples (NOT / sum of the
                        weights); the epoch loss keeps its Mean over batches weighted by batch size
                        (keras/engine/compile_utils.py ``LossesContainer``)
* class_weight          keras/engine/data_adapter.py ``_make_class_weight_map_fn``: keys must be
                        exactly 0 .. K-1 (else ValueError); class = int(y); the class weight is
                        gathered per sample and multiplies the sample weight when both are given
* weighted metrics      keras/metrics.py ``Mean`` / ``MeanMetricWrapper``: sum(w v) / sum(w) with
                        div_no_nan (0 when the weights sum to 0) -- evaluate's accuracy
"""
import numpy as np

from oracle import keras_mlp as km


def sample_weights(z, sample_weight=None, class_weight=None, dtype=np.float32):
    """The per-sample weights Keras trains with: ``sample_weight`` ((N,) or (N, 1), values unchecked)
    times ``class_weight[int(z_i)]``; None when neither is given.  ValueError for class_weight keys
    other than 0 .. K-1, a label without a key, or a bad sample_weight shape."""
    z = np.asarray(z).reshape(-1)
    n = z.shape[0]
    w = None
    if sample_weight is not None:
        sw = np.asarray(sample_weight)
        if sw.shape not in ((n,), (n, 1)):
            raise ValueError(f"sample_weight shape {sw.shape} does not match {n} samples")
        w = sw.reshape(n).astype(dtype)
    if class_weight is not None:
        if sorted(class_weight) != list(range(len(class_weight))):
            raise ValueError(f"class_weight keys must be 0 .. K-1, got {sorted(class_weight)}")
        table = np.array([class_weight[k] for k in range(len(class_weight))], dtype)
        cls = z.astype(np.int64)
        if cls.size and (cls.min() < 0 or cls.max() >= len(table)):
            raise ValueError("a label has no class_weight key")
        w = table[cls] if w is None else w * table[cls]
    return w


def loss_and_weight_grads(weights, acts, Xb, zb, l2=0.0, dtype=np.float32, sample_weight=None):
    """sum(w_i bce_i) / n over the batch (+ the l2 terms of km.loss_and_weight_grads) and its
    gradient wrt every weight; ``sample_weight`` None is km.loss_and_weight_grads itself."""
    if sample_weight is None:
        return km.loss_and_weight_grads(weights, acts, Xb, zb, l2, dtype)
    f = dtype
    assert acts[-1] in ("sigmoid", "linear")
    acts_l = list(acts[:-1]) + ["linear"]
    u, hs = km.forward(weights, acts_l, Xb, dtype, keep=True)
    n = Xb.shape[0]
    z = zb.astype(dtype).reshape(n, 1)
    sw = np.asarray(sample_weight).astype(dtype).reshape(n, 1)
    loss = f(np.sum(sw * km.bce_with_logits(u, z), dtype=dtype) / f(n))
    delta = sw * (km._sigmoid(u) - z) / f(n)
    grads = [None] * len(weights)
    for l in range(len(acts) - 1, -1, -1):
        if l < len(acts) - 1:
            delta = delta * km._act_grad_from_output(acts_l[l], hs[l + 1])
        grads[2 * l] = hs[l].T @ delta
        grads[2 * l + 1] = delta.sum(axis=0)
        if l > 0:
            delta = delta @ weights[2 * l].T
    l2v = km._l2_vector(l2, len(weights))
    if any(l2v):
        reg = f(0)
        for i, w in enumerate(weights):
            if l2v[i]:
                reg += f(l2v[i]) * f(np.sum(w * w, dtype=dtype))
                grads[i] = grads[i] + f(2 * l2v[i]) * w
        loss = f(loss + reg)
    return loss, grads


def fit(weights, acts, X, z, epochs, batch_size, permutations, adam=None, l2=0.0, dtype=np.float32,
        sample_weight=None, class_weight=None):
    """km.fit with every batch's loss sum(w_i bce_i) / batch_n (weights from ``sample_weights``);
    the epoch loss is sum(batch_loss * batch_n) / N as before.  Returns (history_loss, adam_state)."""
    X = np.asarray(X).astype(dtype)
    z = np.asarray(z).astype(dtype)
    N = X.shape[0]
    w = sample_weights(z, sample_weight, class_weight, dtype)
    if adam is None:
        adam = km.AdamState(weights)
    hist = np.zeros(epochs, dtype)
    for e in range(epochs):
        perm = np.asarray(permutations[e])
        tot = dtype(0)
        for s in range(0, N, batch_size):
            idx = perm[s:s + batch_size]
            loss, grads = loss_and_weight_grads(weights, acts, X[idx], z[idx], l2, dtype,
                                                None if w is None else w[idx])
            tot += loss * dtype(len(idx))
            km.adam_apply(weights, grads, adam, dtype)
        hist[e] = tot / dtype(N)
    return hist, adam


def evaluate(weights, acts, X, z, l2=0.0, dtype=np.float32, sample_weight=None, class_weight=None):
    """km.evaluate weighted: loss sum(w_i bce_i) / N (+ l2), accuracy sum(w_i hit_i) / sum(w_i), 0 when
    the weights sum to 0; the output-threshold quirk of km.evaluate stays."""
    X = np.asarray(X).astype(dtype)
    zz = np.asarray(z).astype(dtype)
    w = sample_weights(zz, sample_weight, class_weight, dtype)
    if w is None:
        return km.evaluate(weights, acts, X, zz, l2, dtype=dtype)
    loss, _ = loss_and_weight_grads(weights, acts, X, zz, l2, dtype, w)
    hit = (km.forward(weights, acts, X, dtype)[:, 0] > 0.5).astype(dtype) == zz
    tot = np.sum(w, dtype=dtype)
    acc = np.sum(w * hit, dtype=dtype) / tot if tot != 0 else dtype(0)
    return [float(loss), float(acc)]
