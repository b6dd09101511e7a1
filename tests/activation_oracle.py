"""Keras 2.5 activations selu, softplus, softsign, hard_sigmoid and exponential in NumPy, on top of the
oracle's restatement of the other five (oracle/keras_mlp.py ``_act`` / ``_act_grad_from_output``).
TEST INFRASTRUCTURE ONLY.  [TF-semantics], unpinned like the rest of the Keras half of the oracle;
tests/test_oracle_activations.py checks value, gradients and fits against an independent torch
implementation in fp64.

The TF 2.5 sources each rule restates (paths inside the tensorflow repository at tag v2.5.0; cited from
knowledge of that tree):

* selu          core/kernels/relu_op_functor.h ``Selu``: features < 0 ? scale_alpha (exp(a) - 1) : scale a,
                scale = 1.0507009873554805, scale_alpha = 1.7580993408473768 (= scale * alpha, alpha =
                1.6732632423543772); ``SeluGrad`` takes the OUTPUTS: activations < 0 ?
                g (activations + scale_alpha) : g scale
* softplus      core/kernels/softplus_op.h ``Softplus``: threshold = log(epsilon) + 2 (-13.942385 in fp32);
                a > -threshold ? a : (a < threshold ? exp(a) : log(exp(a) + 1)); ``SoftplusGrad`` takes the
                FEATURES: g / (1 + exp(-a))
* softsign      core/kernels/softsign_op.h ``Softsign``: a / (|a| + 1); ``SoftsignGrad`` takes the
                FEATURES: g / (1 + |a|)^2
* hard_sigmoid  python/keras/backend.py ``hard_sigmoid``: multiply(a, 0.2), add 0.5, clip_by_value(0, 1) --
                three ops, each rounded (not torch's relu6(a + 3) / 6); the gradient of clip_by_value's
                minimum / maximum passes g where 0 <= 0.2 a + 0.5 <= 1 (closed interval)
* exponential   python/keras/activations.py ``exponential`` = math_ops.exp; the ``Exp`` gradient is g y

The kernels keep only the layer output h, so their backward pass uses d act / d a as a function of h
(``act_grad_from_output``): exact for selu and exponential; for softplus (-expm1(-h)), softsign
((1 - |h|)^2) and hard_sigmoid (0.2 on the open interval 0 < h < 1) it differs from TF's features-based
rule (``act_grad_from_features``) by rounding, and for hard_sigmoid at its two edges.  The oracle's
backward pass follows the kernels; DESIGN.md ("Activations") gives the measured deviation from TF's rule.
"""
import contextlib

import numpy as np

from oracle import keras_mlp as km

NEW = ("selu", "softplus", "softsign", "hard_sigmoid", "exponential")
ACTIVATIONS = tuple(km.ACTIVATIONS) + NEW

SELU_SCALE = 1.0507009873554805
SELU_SCALE_ALPHA = 1.7580993408473768


def softplus_threshold(dtype):
    """softplus_op.h: log(epsilon) + 2 in the op's dtype."""
    f = np.dtype(dtype).type
    return f(f(np.log(np.finfo(dtype).eps)) + f(2))


def act(name, a):
    """Forward of every Keras activation the kernels take, in a's dtype."""
    if name not in NEW:
        return _KM_ACT(name, a)
    f = a.dtype.type
    if name == "selu":
        return np.where(a > 0, f(SELU_SCALE) * a, f(SELU_SCALE_ALPHA) * np.expm1(np.minimum(a, f(0))))
    if name == "softplus":
        thr = softplus_threshold(a.dtype)
        with np.errstate(over="ignore"):
            e = np.exp(a)
            return np.where(a > -thr, a, np.where(a < thr, e, np.log(e + f(1))))
    if name == "softsign":
        return a / (np.abs(a) + f(1))
    if name == "hard_sigmoid":
        return np.clip(a * f(0.2) + f(0.5), f(0), f(1))
    if name == "exponential":
        return np.exp(a)


def act_grad_from_output(name, h):
    """d act / d pre-activation through the layer output h: the rule of csrc/act.cuh."""
    if name not in NEW:
        return _KM_GRAD(name, h)
    f = h.dtype.type
    if name == "selu":
        return np.where(h < 0, h + f(SELU_SCALE_ALPHA), f(SELU_SCALE)).astype(h.dtype)
    if name == "softplus":
        return -np.expm1(-h)
    if name == "softsign":
        t = f(1) - np.abs(h)
        return t * t
    if name == "hard_sigmoid":
        return np.where((h > 0) & (h < 1), f(0.2), f(0)).astype(h.dtype)
    if name == "exponential":
        return h.copy()


def act_grad_from_features(name, a):
    """TF's own gradient rule, from the pre-activation a (only the three that TF takes from the features)."""
    f = a.dtype.type
    if name == "softplus":
        return f(1) / (f(1) + np.exp(-a))
    if name == "softsign":
        t = f(1) + np.abs(a)
        return f(1) / (t * t)
    if name == "hard_sigmoid":
        x = a * f(0.2) + f(0.5)
        return np.where((x >= 0) & (x <= 1), f(0.2), f(0)).astype(a.dtype)
    raise ValueError(name)


_KM_ACT, _KM_GRAD = km._act, km._act_grad_from_output


@contextlib.contextmanager
def installed():
    """Every oracle module (keras_mlp, keras_lstm, argmax, svgd) takes the new names while this is open;
    the other five keep the oracle's own functions."""
    saved = km._act, km._act_grad_from_output
    km._act, km._act_grad_from_output = act, act_grad_from_output
    try:
        yield
    finally:
        km._act, km._act_grad_from_output = saved
