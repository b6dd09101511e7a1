"""Keras 2.5 l1 and l1_l2 regularisation for the oracle fit loops (oracle/keras_mlp.py, oracle/keras_lstm.py),
which stay unchanged.  TEST INFRASTRUCTURE ONLY.

[TF-semantics], unpinned like the rest of the oracle: restates keras/regularizers.py of TF 2.5 from knowledge of its
source.

* ``L1(l1=0.01)`` adds ``l1 * reduce_sum(abs(x))``; ``L2(l2=0.01)`` adds ``l2 * reduce_sum(square(x))``.
* ``L1L2(l1=0., l2=0.)`` adds ``l1 * sum|x| + l2 * sum x^2``, each term only when its factor is non-zero.
* The gradient of ``abs`` is TF's ``Abs`` gradient, ``sign(x)``, with sign(0) = 0: a parameter at exactly 0 gets no
  l1 gradient (every bias on the first step).
* The penalty enters the training loss on the values before the step's update, and ``evaluate``'s loss.

``installed()`` wraps ``loss_and_weight_grads`` of both oracle modules and of tests/weighted_oracle.py -- the name
their fit loops (and the MLP ``evaluate``s) call -- so that a ``Factors`` passed as their ``l2`` argument adds the l1
terms on top of the oracle's own l2 rule.  Anything else passed as ``l2`` reaches the oracle unchanged.
"""
import contextlib

import numpy as np

from oracle import keras_lstm as kl, keras_mlp as km
import weighted_oracle as wo


class Factors:
    """Per-array l2 and l1 factors in Keras weight order (scalars: the same factor for every array)."""

    def __init__(self, l2=0.0, l1=0.0):
        self.l2, self.l1 = l2, l1


def l1_penalty(weights, l1):
    """sum_i l1_i * sum|w_i| in fp64 (the evaluate loss's l1 term)."""
    l1v = km._l2_vector(l1, len(weights))
    return float(sum(f * np.sum(np.abs(w), dtype=np.float64) for f, w in zip(l1v, weights) if f))


def _with_l1(loss, grads, weights, l1, f):
    l1v = km._l2_vector(l1, len(weights))
    if not any(l1v):
        return loss, grads
    reg = f(0)
    for i, w in enumerate(weights):
        if l1v[i]:
            reg += f(l1v[i]) * f(np.sum(np.abs(w), dtype=f))
            grads[i] = grads[i] + f(l1v[i]) * np.sign(w).astype(f)  # np.sign(0) == 0
    return f(loss + reg), grads


_KM_LOSS, _KL_LOSS, _WO_LOSS = km.loss_and_weight_grads, kl.loss_and_weight_grads, wo.loss_and_weight_grads


def _km_loss(weights, acts, Xb, zb, l2=0.0, dtype=np.float32):
    if not isinstance(l2, Factors):
        return _KM_LOSS(weights, acts, Xb, zb, l2, dtype)
    loss, grads = _KM_LOSS(weights, acts, Xb, zb, l2.l2, dtype)
    return _with_l1(loss, grads, weights, l2.l1, dtype)


def _kl_loss(weights, activation, Xb, Yb, mask, l2=None, dtype=np.float32):
    if not isinstance(l2, Factors):
        return _KL_LOSS(weights, activation, Xb, Yb, mask, l2, dtype)
    loss, grads = _KL_LOSS(weights, activation, Xb, Yb, mask, l2.l2, dtype)
    return _with_l1(loss, grads, weights, l2.l1, dtype)


def _wo_loss(weights, acts, Xb, zb, l2=0.0, dtype=np.float32, sample_weight=None):
    if not isinstance(l2, Factors) or sample_weight is None:  # unweighted: km's function, wrapped above
        return _WO_LOSS(weights, acts, Xb, zb, l2, dtype, sample_weight)
    loss, grads = _WO_LOSS(weights, acts, Xb, zb, l2.l2, dtype, sample_weight)
    return _with_l1(loss, grads, weights, l2.l1, dtype)


def lstm_evaluate(weights, activation, X, Y, mask_value, factors, dtype=np.float32):
    """``kl.evaluate`` with the l1 penalty added to the loss."""
    out = kl.evaluate(weights, activation, X, Y, mask_value, l2=factors.l2, dtype=dtype)
    return [out[0] + l1_penalty(weights, factors.l1), out[1]]


@contextlib.contextmanager
def installed():
    saved = km.loss_and_weight_grads, kl.loss_and_weight_grads, wo.loss_and_weight_grads
    km.loss_and_weight_grads, kl.loss_and_weight_grads, wo.loss_and_weight_grads = _km_loss, _kl_loss, _wo_loss
    try:
        yield
    finally:
        km.loss_and_weight_grads, kl.loss_and_weight_grads, wo.loss_and_weight_grads = saved
