"""Keras 2.5 learning-rate schedules for the oracle fit loops (oracle/keras_mlp.py, oracle/keras_lstm.py), which stay
unchanged.  TEST INFRASTRUCTURE ONLY.

[TF-semantics], unpinned like the rest of the oracle: each schedule restates TF 2.5 from knowledge of its source,
keras/optimizer_v2/learning_rate_schedule.py, in np.float32 (the dtype of a float initial_learning_rate; every
operand is cast to it, each operation rounds on its own):

* ExponentialDecay        p = step / decay_steps, floor(p) if staircase; initial * pow(decay_rate, p)
* InverseTimeDecay        p as above; initial / (1 + decay_rate * p)
* PolynomialDecay         cycle: decay_steps * (1 if step == 0 else ceil(step / decay_steps)), else
                          step = min(step, decay_steps); (initial - end) * pow(1 - step / decay_steps', power) + end
* PiecewiseConstantDecay  values[0] if step <= b_0, values[i + 1] if b_i < step <= b_{i+1}, values[-1] if
                          step > b_last; the boundaries are cast to the step's dtype (float32)

keras/optimizer_v2/optimizer_v2.py ``_decayed_lr`` evaluates the schedule at ``cast(self.iterations, float32)``
before ``apply_gradients`` increments it: update t (1-based) uses the schedule at t - 1.

``installed(schedule)`` wraps ``km.adam_apply`` -- the name both oracle fit loops call, also when
``optimizer_oracle.installed()`` has replaced it -- so that the state's ``lr`` is the schedule at ``state.t`` (still
t - 1: every rule increments t itself) before each update.
"""
import contextlib
import math

import numpy as np

from oracle import keras_mlp as km

f32 = np.float32


def exponential(step, initial_learning_rate, decay_steps, decay_rate, staircase=False, name=None):
    p = f32(step) / f32(decay_steps)
    if staircase:
        p = np.floor(p)
    return f32(initial_learning_rate) * np.power(f32(decay_rate), p)


def inverse_time(step, initial_learning_rate, decay_steps, decay_rate, staircase=False, name=None):
    p = f32(step) / f32(decay_steps)
    if staircase:
        p = np.floor(p)
    return f32(initial_learning_rate) / (f32(1) + f32(decay_rate) * p)


def polynomial(step, initial_learning_rate, decay_steps, end_learning_rate=1e-4, power=1.0, cycle=False, name=None):
    s, ds = f32(step), f32(decay_steps)
    if cycle:
        ds = ds * (f32(1) if s == 0 else np.ceil(s / f32(decay_steps)))
    else:
        s = np.minimum(s, ds)
    return ((f32(initial_learning_rate) - f32(end_learning_rate)) * np.power(f32(1) - s / ds, f32(power))
            + f32(end_learning_rate))


def piecewise(step, boundaries, values, name=None):
    s = f32(step)
    if s <= f32(boundaries[0]):
        return f32(values[0])
    if s > f32(boundaries[-1]):
        return f32(values[-1])
    for lo, hi, v in zip(boundaries[:-1], boundaries[1:], values[1:-1]):
        if f32(lo) < s <= f32(hi):
            return f32(v)
    raise AssertionError("unreachable")


def exact(step, kind, **cfg):
    """The same schedules in float64 Python arithmetic, for the rounding check."""
    s = float(step)
    if kind == "piecewise":
        b, v = cfg["boundaries"], cfg["values"]
        return float(v[sum(s > x for x in b)])
    ds = float(cfg["decay_steps"])
    if kind == "polynomial":
        if cfg.get("cycle", False):
            ds = ds * (1.0 if s == 0 else math.ceil(s / ds))
        else:
            s = min(s, ds)
        ini, end = float(cfg["initial_learning_rate"]), float(cfg.get("end_learning_rate", 1e-4))
        return (ini - end) * (1.0 - s / ds) ** float(cfg.get("power", 1.0)) + end
    p = s / ds
    if cfg.get("staircase", False):
        p = math.floor(p)
    if kind == "exponential":
        return float(cfg["initial_learning_rate"]) * float(cfg["decay_rate"]) ** p
    return float(cfg["initial_learning_rate"]) / (1.0 + float(cfg["decay_rate"]) * p)


_KIND = {"ExponentialDecay": exponential, "InverseTimeDecay": inverse_time, "PolynomialDecay": polynomial,
         "PiecewiseConstantDecay": piecewise}


def rate(schedule):
    """step -> float32 rate of a ``bore_b200.schedules`` object, through this module's restatement of its class
    and its ``get_config()``."""
    fn, cfg = _KIND[type(schedule).__name__], schedule.get_config()
    return lambda step: fn(step, **cfg)


@contextlib.contextmanager
def installed(schedule):
    fn = rate(schedule)
    inner = km.adam_apply

    def apply(weights, grads, st, dtype=np.float32):
        st.lr = float(fn(st.t))
        return inner(weights, grads, st, dtype)

    km.adam_apply = apply
    try:
        yield
    finally:
        km.adam_apply = inner
