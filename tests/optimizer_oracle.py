"""Keras 2.5 optimizers RMSprop, Adagrad, Adadelta, Adamax and Nadam for the oracle fit loops
(oracle/keras_mlp.py, oracle/keras_lstm.py), which stay unchanged.  TEST INFRASTRUCTURE ONLY.

[TF-semantics], unpinned like the rest of the oracle: each rule restates TF 2.5 from knowledge of its source.
``g`` is the gradient with the l2 term, ``t`` is Keras' ``iterations + 1``; every slot starts at zero unless said.

* RMSprop   keras/optimizer_v2/rmsprop.py.  momentum = 0 takes the Python path of ``_resource_apply_dense``:
            rms = rho rms + (1 - rho) g^2; centered: mg = rho mg + (1 - rho) g, denom = rms - mg^2, else
            denom = rms; w -= lr g / (sqrt(denom) + eps).  momentum > 0 (not centered) calls
            ResourceApplyRMSProp (core/kernels/training_ops.cc ``ApplyRMSProp``): ms += (g^2 - ms)(1 - rho);
            mom = momentum mom + lr g / sqrt(ms + eps); w -= mom -- eps INSIDE the root.
* Adagrad   keras/optimizer_v2/adagrad.py -> ResourceApplyAdagradV2 (``ApplyAdagradV2``): the accumulator
            starts at initial_accumulator_value; acc += g^2; w -= lr g / (sqrt(acc) + eps).
* Adadelta  keras/optimizer_v2/adadelta.py -> ResourceApplyAdadelta (``ApplyAdadelta``):
            a = rho a + (1 - rho) g^2; u = sqrt(av + eps) / sqrt(a + eps) g; av = rho av + (1 - rho) u^2;
            w -= lr u.
* Adamax    keras/optimizer_v2/adamax.py -> ResourceApplyAdaMax (``ApplyAdaMax``): m += (g - m)(1 - b1);
            v = max(b2 v, |g|); w -= lr / (1 - b1^t) m / (v + eps).
* Nadam     keras/optimizer_v2/nadam.py ``_prepare_local`` / ``_resource_apply_dense``:
            mu_t = b1 (1 - 0.5 0.96^(0.004 t)), mu_{t+1} likewise; cache <- cache mu_t (the m_cache variable,
            starts at 1); m = b1 m + (1 - b1) g; v = b2 v + (1 - b2) g^2;
            mbar = (1 - mu_t) g / (1 - cache) + mu_{t+1} m / (1 - cache mu_{t+1});
            w -= lr mbar / (sqrt(v / (1 - b2^t)) + eps).  The learning rate is not decayed.

``installed()`` makes ``km.adam_apply`` -- the name both oracle fit loops call -- dispatch on the state's type;
``km.AdamState`` states still reach the oracle's own Adam.
"""
import contextlib

import numpy as np

from oracle import keras_mlp as km


class _State:
    def __init__(self, weights, s0=0.0):
        self.s0 = [np.full_like(w, s0) for w in weights]
        self.s1 = [np.zeros_like(w) for w in weights]
        self.t = 0


class RMSpropState(_State):
    def __init__(self, weights, lr=1e-3, rho=0.9, momentum=0.0, eps=1e-7, centered=False):
        super().__init__(weights)
        self.lr, self.rho, self.momentum, self.eps, self.centered = lr, rho, momentum, eps, centered

    def apply(self, weights, grads, f):
        rho, lr, eps = f(self.rho), f(self.lr), f(self.eps)
        for i, g in enumerate(grads):
            if self.momentum > 0:
                self.s0[i] += (g * g - self.s0[i]) * (f(1) - rho)
                self.s1[i] = f(self.momentum) * self.s1[i] + lr * g / np.sqrt(self.s0[i] + eps)
                weights[i] -= self.s1[i]
                continue
            self.s0[i] = rho * self.s0[i] + (f(1) - rho) * (g * g)
            den = self.s0[i]
            if self.centered:
                self.s1[i] = rho * self.s1[i] + (f(1) - rho) * g
                den = self.s0[i] - self.s1[i] * self.s1[i]
            weights[i] -= lr * g / (np.sqrt(den) + eps)


class AdagradState(_State):
    def __init__(self, weights, lr=1e-3, initial_accumulator_value=0.1, eps=1e-7):
        super().__init__(weights, initial_accumulator_value)
        self.lr, self.eps = lr, eps

    def apply(self, weights, grads, f):
        for i, g in enumerate(grads):
            self.s0[i] += g * g
            weights[i] -= f(self.lr) * g / (np.sqrt(self.s0[i]) + f(self.eps))


class AdadeltaState(_State):
    def __init__(self, weights, lr=1e-3, rho=0.95, eps=1e-7):
        super().__init__(weights)
        self.lr, self.rho, self.eps = lr, rho, eps

    def apply(self, weights, grads, f):
        rho, eps = f(self.rho), f(self.eps)
        for i, g in enumerate(grads):
            self.s0[i] = self.s0[i] * rho + (g * g) * (f(1) - rho)
            u = np.sqrt(self.s1[i] + eps) / np.sqrt(self.s0[i] + eps) * g
            self.s1[i] = self.s1[i] * rho + (u * u) * (f(1) - rho)
            weights[i] -= u * f(self.lr)


class AdamaxState(_State):
    def __init__(self, weights, lr=1e-3, beta1=0.9, beta2=0.999, eps=1e-7):
        super().__init__(weights)
        self.lr, self.beta1, self.beta2, self.eps = lr, beta1, beta2, eps

    def apply(self, weights, grads, f):
        b1 = f(self.beta1)
        step = f(self.lr) / (f(1) - f(np.power(b1, f(self.t))))
        for i, g in enumerate(grads):
            self.s0[i] += (g - self.s0[i]) * (f(1) - b1)
            self.s1[i] = np.maximum(f(self.beta2) * self.s1[i], np.abs(g))
            weights[i] -= step * (self.s0[i] / (self.s1[i] + f(self.eps)))


class NadamState(_State):
    def __init__(self, weights, lr=1e-3, beta1=0.9, beta2=0.999, eps=1e-7):
        super().__init__(weights)
        self.lr, self.beta1, self.beta2, self.eps = lr, beta1, beta2, eps
        self.cache = 1.0

    def apply(self, weights, grads, f):
        b1, b2 = f(self.beta1), f(self.beta2)
        mu = b1 * (f(1) - f(0.5) * f(np.power(f(0.96), f(0.004) * f(self.t))))
        mu_next = b1 * (f(1) - f(0.5) * f(np.power(f(0.96), f(0.004) * f(self.t + 1))))
        self.cache = f(self.cache) * mu
        vd = f(1) - f(np.power(b2, f(self.t)))
        for i, g in enumerate(grads):
            self.s0[i] = b1 * self.s0[i] + (f(1) - b1) * g
            self.s1[i] = b2 * self.s1[i] + (f(1) - b2) * (g * g)
            mbar = (f(1) - mu) * g / (f(1) - self.cache) + mu_next * self.s0[i] / (f(1) - self.cache * mu_next)
            weights[i] -= f(self.lr) * mbar / (np.sqrt(self.s1[i] / vd) + f(self.eps))


def state_for(weights, optimizer, dtype=np.float32):
    """The oracle state of a ``bore_b200.layers`` optimizer object (``km.AdamState`` for Adam)."""
    o, f = optimizer, dtype
    kind = o.kind
    if kind == "adam":
        return km.AdamState(weights, o.learning_rate, o.beta_1, o.beta_2, o.epsilon)
    if kind == "rmsprop":
        st = RMSpropState(weights, o.learning_rate, o.rho, o.momentum, o.epsilon, o.centered)
    elif kind == "adagrad":
        st = AdagradState(weights, o.learning_rate, o.initial_accumulator_value, o.epsilon)
    elif kind == "adadelta":
        st = AdadeltaState(weights, o.learning_rate, o.rho, o.epsilon)
    elif kind == "adamax":
        st = AdamaxState(weights, o.learning_rate, o.beta_1, o.beta_2, o.epsilon)
    else:
        st = NadamState(weights, o.learning_rate, o.beta_1, o.beta_2, o.epsilon)
    st.s0 = [s.astype(f) for s in st.s0]
    st.s1 = [s.astype(f) for s in st.s1]
    return st


_KM_ADAM = km.adam_apply


def apply(weights, grads, st, dtype=np.float32):
    """``km.adam_apply`` while ``installed()``: the rule of ``st``'s kind."""
    if isinstance(st, km.AdamState):
        return _KM_ADAM(weights, grads, st, dtype)
    st.t += 1
    st.apply(weights, grads, dtype)


@contextlib.contextmanager
def installed():
    saved = km.adam_apply
    km.adam_apply = apply
    try:
        yield
    finally:
        km.adam_apply = saved
