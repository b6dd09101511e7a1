"""Keras 2.5 learning-rate schedules the training kernels evaluate on the device (``keras.optimizers.schedules``).

An optimizer of ``bore_b200.layers`` takes an instance of one of the four classes below as its
``learning_rate``.  Update number t of a model (1-based) uses ``schedule(t - 1)``: Keras' ``_decayed_lr``
evaluates the schedule at ``iterations`` before the increment, so a later ``fit`` continues the schedule.
``__call__`` gives the rate of a step in float32, the arithmetic of the kernels (DESIGN.md, "Learning-rate
schedules")."""

import numpy as np

# schedule codes of the training kernels (include/bore_b200.h, BORE_LR_*)
LR_CODES = {"constant": 0, "exponential": 1, "inverse_time": 2, "polynomial": 3, "piecewise": 4}
MAX_BOUNDARIES = 16  # BORE_LR_MAX_BOUNDARIES

_f32 = np.float32


class LearningRateSchedule:
    """``keras.optimizers.schedules.LearningRateSchedule``.  Only the four classes of this module reach the
    kernels: an optimizer refuses a subclass, since its ``__call__`` is Python."""

    code = None

    def __call__(self, step):
        raise NotImplementedError("LearningRateSchedule is a base class")

    def get_config(self):
        raise NotImplementedError("LearningRateSchedule is a base class")

    def native(self):
        """(BORE_LR_* code, the parameters of bore_mlp_set_lr_schedule); ValueError for arguments the kernels
        do not take (a non-finite value, decay_steps <= 0, boundaries not strictly increasing or more than
        16 of them), raised when the optimizer is made rather than at the first fit."""
        code, sp = self._native()
        if not all(np.isfinite(_f32(v)) for v in sp):
            raise ValueError(f"{type(self).__name__}: every argument must be finite, got {self.get_config()}")
        return code, sp


class _Decay(LearningRateSchedule):
    """The schedules with ``decay_steps``."""

    def _decay_steps_ok(self):
        if not _f32(self.decay_steps) > 0:
            raise ValueError(f"{type(self).__name__}: decay_steps must be > 0, got {self.decay_steps!r} (Keras "
                             "would give NaN or inf rates)")


class ExponentialDecay(_Decay):
    """``initial_learning_rate * decay_rate ** (step / decay_steps)``, the exponent floored when ``staircase``."""

    code = LR_CODES["exponential"]

    def __init__(self, initial_learning_rate, decay_steps, decay_rate, staircase=False, name=None):
        self.initial_learning_rate = initial_learning_rate
        self.decay_steps = decay_steps
        self.decay_rate = decay_rate
        self.staircase = staircase
        self.name = name

    def __call__(self, step):
        p = _f32(step) / _f32(self.decay_steps)
        if self.staircase:
            p = np.floor(p)
        return _f32(self.initial_learning_rate) * np.power(_f32(self.decay_rate), p)

    def get_config(self):
        return {"initial_learning_rate": self.initial_learning_rate, "decay_steps": self.decay_steps,
                "decay_rate": self.decay_rate, "staircase": self.staircase, "name": self.name}

    def _native(self):
        self._decay_steps_ok()
        return self.code, [float(self.initial_learning_rate), float(self.decay_steps), float(self.decay_rate),
                           float(bool(self.staircase))]


class InverseTimeDecay(_Decay):
    """``initial_learning_rate / (1 + decay_rate * step / decay_steps)``, ``step / decay_steps`` floored when
    ``staircase``."""

    code = LR_CODES["inverse_time"]

    def __init__(self, initial_learning_rate, decay_steps, decay_rate, staircase=False, name=None):
        self.initial_learning_rate = initial_learning_rate
        self.decay_steps = decay_steps
        self.decay_rate = decay_rate
        self.staircase = staircase
        self.name = name

    def __call__(self, step):
        p = _f32(step) / _f32(self.decay_steps)
        if self.staircase:
            p = np.floor(p)
        return _f32(self.initial_learning_rate) / (_f32(1) + _f32(self.decay_rate) * p)

    def get_config(self):
        return {"initial_learning_rate": self.initial_learning_rate, "decay_steps": self.decay_steps,
                "decay_rate": self.decay_rate, "staircase": self.staircase, "name": self.name}

    def _native(self):
        self._decay_steps_ok()
        return self.code, [float(self.initial_learning_rate), float(self.decay_steps), float(self.decay_rate),
                           float(bool(self.staircase))]


class PolynomialDecay(_Decay):
    """``(initial - end) * (1 - step / decay_steps) ** power + end`` with the step clamped at ``decay_steps``;
    with ``cycle``, ``decay_steps`` is multiplied by ``ceil(step / decay_steps)`` (1 at step 0) instead."""

    code = LR_CODES["polynomial"]

    def __init__(self, initial_learning_rate, decay_steps, end_learning_rate=0.0001, power=1.0, cycle=False,
                 name=None):
        self.initial_learning_rate = initial_learning_rate
        self.decay_steps = decay_steps
        self.end_learning_rate = end_learning_rate
        self.power = power
        self.cycle = cycle
        self.name = name

    def __call__(self, step):
        s, ds = _f32(step), _f32(self.decay_steps)
        if self.cycle:
            ds = ds * (_f32(1) if s == 0 else np.ceil(s / ds))
        else:
            s = np.minimum(s, ds)
        ini, end = _f32(self.initial_learning_rate), _f32(self.end_learning_rate)
        return (ini - end) * np.power(_f32(1) - s / ds, _f32(self.power)) + end

    def get_config(self):
        return {"initial_learning_rate": self.initial_learning_rate, "decay_steps": self.decay_steps,
                "end_learning_rate": self.end_learning_rate, "power": self.power, "cycle": self.cycle,
                "name": self.name}

    def _native(self):
        self._decay_steps_ok()
        return self.code, [float(self.initial_learning_rate), float(self.decay_steps),
                           float(self.end_learning_rate), float(self.power), float(bool(self.cycle))]


class PiecewiseConstantDecay(LearningRateSchedule):
    """``values[0]`` for ``step <= boundaries[0]``, ``values[i + 1]`` for ``boundaries[i] < step <=
    boundaries[i + 1]``, ``values[-1]`` past the last boundary; the boundaries are compared in float32, the
    step's dtype."""

    code = LR_CODES["piecewise"]

    def __init__(self, boundaries, values, name=None):
        if len(boundaries) != len(values) - 1:
            raise ValueError("The length of boundaries should be 1 less than the length of values")
        self.boundaries = boundaries
        self.values = values
        self.name = name

    def __call__(self, step):
        s = _f32(step)
        i = 0
        while i < len(self.boundaries) and s > _f32(self.boundaries[i]):
            i += 1
        return _f32(self.values[i])

    def get_config(self):
        return {"boundaries": self.boundaries, "values": self.values, "name": self.name}

    def _native(self):
        b = [float(_f32(v)) for v in self.boundaries]
        if not 1 <= len(b) <= MAX_BOUNDARIES:
            raise ValueError(f"PiecewiseConstantDecay: 1 to {MAX_BOUNDARIES} boundaries are taken, got {len(b)}")
        if any(hi <= lo for lo, hi in zip(b, b[1:])):
            raise ValueError(f"PiecewiseConstantDecay: boundaries must be strictly increasing in float32, got "
                             f"{self.boundaries!r}")
        return self.code, b + [float(v) for v in self.values]


SCHEDULES = (ExponentialDecay, InverseTimeDecay, PolynomialDecay, PiecewiseConstantDecay)
