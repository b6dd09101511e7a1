"""Keras-shaped declarations the hot path needs: Dense, the regularizers, BinaryCrossentropy and the optimizers.

Keras itself is absent (and not wanted on the path); these are plain spec objects that
``bore_b200.models.Sequential`` lowers onto the native handle.  Names and arguments follow
the call sites README.rst:60-66 and bore/plugins/hpbandster/base.py:113-116,147-158."""

import numpy as np

from . import schedules

# Keras 2.5 element-wise activations whose derivative is a function of the layer output, the one value the
# kernels keep (swish and gelu are not: DESIGN.md, "Activations")
_ACTIVATIONS = ("linear", "relu", "elu", "sigmoid", "tanh", "selu", "softplus", "softsign", "hard_sigmoid",
                "exponential")


def activation_name(activation, owner):
    """The Keras name of ``activation`` (a name, a Keras-named callable or None, which is linear);
    ValueError naming the accepted ones for any other."""
    if callable(activation):
        activation = getattr(activation, "__name__", activation)
    if activation is None:
        activation = "linear"
    if activation not in _ACTIVATIONS:
        raise ValueError(f"{owner}: activation must be one of {_ACTIVATIONS}, got {activation!r}")
    return activation


def _penalty(value, owner):
    """A regularisation factor the kernels take: a finite number >= 0."""
    v = float(value)
    if not np.isfinite(v) or v < 0:
        raise ValueError(f"{owner}: the regularisation factor must be finite and >= 0, got {value!r}")
    return v


class L1:
    """``keras.regularizers.L1(l1=0.01)``: adds ``l1 * sum(abs(w))`` to the loss; its gradient is
    ``l1 * sign(w)`` with sign(0) = 0 (TF's Abs gradient)."""

    def __init__(self, l1=0.01):
        self.l1 = _penalty(0.01 if l1 is None else l1, "L1")


class L2:
    """``keras.regularizers.l2(l2)``: adds ``l2 * sum(w**2)`` to the loss."""

    def __init__(self, l2=0.01):
        self.l2 = float(l2)


class L1L2:
    """``keras.regularizers.L1L2(l1=0., l2=0.)``: adds ``l1 * sum(abs(w)) + l2 * sum(w**2)``, each term only
    when its factor is non-zero.  Its defaults are zeros; ``l1_l2()`` and the string ``"l1_l2"`` give 0.01 each."""

    def __init__(self, l1=0.0, l2=0.0):
        self.l1 = _penalty(0.0 if l1 is None else l1, "L1L2")
        self.l2 = _penalty(0.0 if l2 is None else l2, "L1L2")


l1 = L1


def l2(l2=0.01):
    return L2(l2)


def l1_l2(l1=0.01, l2=0.01):
    """``keras.regularizers.l1_l2``: ``L1L2`` with 0.01 for each factor by default."""
    return L1L2(l1=l1, l2=l2)


# keras.regularizers.get / deserialize: the strings it takes and what they give ("l1_l2" is deserialize's special
# case, L1L2(0.01, 0.01), not the class's zeros)
_REGULARIZER_NAMES = {"l1": L1, "L1": L1, "l2": L2, "L2": L2, "L1L2": L1L2, "l1_l2": l1_l2}


def regularizer_get(identifier, owner):
    """``keras.regularizers.get``: None, an ``L1`` / ``L2`` / ``L1L2`` instance, or one of the names
    ``"l1"``, ``"l2"``, ``"L1"``, ``"L2"``, ``"L1L2"`` (class defaults) and ``"l1_l2"`` (0.01 each).
    ValueError naming what is accepted for anything else: the kernels apply no other penalty."""
    if identifier is None or isinstance(identifier, (L1, L2, L1L2)):
        return identifier
    if isinstance(identifier, str) and identifier in _REGULARIZER_NAMES:
        return _REGULARIZER_NAMES[identifier]()
    raise ValueError(f"{owner}: a regularizer must be None, an instance of bore_b200.layers.{{L1, L2, L1L2}} "
                     f"or one of the names {tuple(_REGULARIZER_NAMES)}, got {identifier!r}")


def regularizer_factors(regularizers):
    """The per-array (l2, l1) factor lists of a sequence of regularizers, as the native setters take them
    (None: no penalty)."""
    regularizers = list(regularizers)
    l2s = [0.0 if r is None else float(getattr(r, "l2", 0.0)) for r in regularizers]
    l1s = [0.0 if r is None else float(getattr(r, "l1", 0.0)) for r in regularizers]
    return l2s, l1s


class Dense:
    """``keras.layers.Dense(units, activation=None, input_dim=None, kernel_regularizer=None,
    bias_regularizer=None)``: ``y = act(x @ W + b)``, glorot-uniform kernel, zero bias."""

    def __init__(self, units, activation=None, input_dim=None, input_shape=None,
                 kernel_regularizer=None, bias_regularizer=None, use_bias=True, **kwargs):
        if kwargs:
            raise TypeError(f"Dense: unsupported arguments {sorted(kwargs)}")
        if not use_bias:
            raise NotImplementedError("Dense(use_bias=False) is not on the BORE-MLP path")
        activation = activation_name(activation, "Dense")
        if input_shape is not None and input_dim is None:
            (input_dim,) = input_shape
        self.units = int(units)
        self.activation = activation
        self.input_dim = None if input_dim is None else int(input_dim)
        self.kernel_regularizer = regularizer_get(kernel_regularizer, "Dense")
        self.bias_regularizer = regularizer_get(bias_regularizer, "Dense")


class Dropout:
    """``keras.layers.Dropout(rate, noise_shape=None, seed=None)``: in training, each unit of the layer's input is
    kept with probability 1 - rate and scaled by 1 / (1 - rate); ``predict`` and ``evaluate`` see no dropout.  Only
    directly after a hidden ``Dense`` layer.  ``rate`` must be finite and in [0, 1), checked here rather than at the
    first call as Keras does; ``seed`` is a uint32, or None for one drawn from the model's ``RandomState`` when its
    weights are made.  The mask is the project's own (DESIGN.md, "Dropout"): TF's random stream is not reproduced."""

    def __init__(self, rate, noise_shape=None, seed=None, **kwargs):
        if kwargs:
            raise TypeError(f"Dropout: unsupported arguments {sorted(kwargs)}")
        if noise_shape is not None:
            raise NotImplementedError("Dropout(noise_shape=...) is not in the training kernels: their masks are per "
                                      "sample and unit")
        r = float(rate)
        if not (np.isfinite(r) and 0.0 <= r < 1.0):
            raise ValueError(f"Dropout: rate must be finite and in [0, 1), got {rate!r}")
        if seed is not None and not (int(seed) == seed and 0 <= int(seed) < 2 ** 32):
            raise ValueError(f"Dropout: seed must be None or an integer in [0, 2**32), got {seed!r}")
        self.rate = r
        self.noise_shape = None
        self.seed = None if seed is None else int(seed)


def split_dropout(layers, final=True):
    """(the Dense layers, the Dropout after each hidden layer or None) of a layer list.  A Dropout is taken only
    directly after a hidden Dense layer; NotImplementedError says why for any other place.  ``final=False``: the list
    may still grow (``add``), so its last Dense layer need not be the output layer, and ``after`` has an entry for it."""
    dense, after = [], []
    for lyr in layers:
        check_layer_order(dense, after, lyr)
        if isinstance(lyr, Dense):
            dense.append(lyr)
            after.append(None)
        else:
            after[-1] = lyr
    if not final:
        return dense, after
    if after and after[-1] is not None:
        raise NotImplementedError("a Dropout must be followed by a Dense layer: dropout after the output layer is "
                                  "not taken, since the loss reaches through to its logit")
    return dense, after[:-1]


def check_layer_order(dense, after, layer):
    """What ``add`` can check of appending ``layer`` to the Dense layers ``dense`` with their Dropouts ``after``."""
    if isinstance(layer, Dense):
        return
    if not isinstance(layer, Dropout):
        raise NotImplementedError("only Dense and Dropout layers are on the BORE-MLP path")
    if not dense:
        raise NotImplementedError("a Dropout as the first layer (input dropout) is not taken: the training kernels "
                                  "gather the minibatch straight into their tiles")
    if after[-1] is not None:
        raise NotImplementedError("two Dropout layers in a row are not taken: a Dropout must follow a Dense layer")


def dropout_rates_seeds(after, random_state):
    """The (rates, seeds) of the hidden layers for ``NativeMLP.set_dropout``, or None when no rate is > 0.  A
    Dropout with ``seed=None`` and rate > 0 draws its seed from ``random_state``, in layer order."""
    if not any(d is not None and d.rate > 0 for d in after):
        return None
    rates, seeds = [], []
    for d in after:
        on = d is not None and d.rate > 0
        rates.append(d.rate if on else 0.0)
        seeds.append(0 if not on else d.seed if d.seed is not None else int(random_state.randint(0, 2 ** 32,
                                                                                                  dtype=np.int64)))
    return rates, seeds


class BinaryCrossentropy:
    """``keras.losses.BinaryCrossentropy(from_logits=...)`` (plugins/hpbandster/base.py:157)."""

    def __init__(self, from_logits=False):
        self.from_logits = bool(from_logits)


# Keras optimizer codes of the training kernels (include/bore_b200.h, BORE_OPT_*)
OPT_CODES = {"adam": 0, "rmsprop": 1, "adagrad": 2, "adadelta": 3, "adamax": 4, "nadam": 5}
# Keras optimizers without a kernel, and why
_OPT_REFUSED = {
    "sgd": "SGD has no training kernel yet",
    "ftrl": "Ftrl has no training kernel (its linear and accumulator slots and l1 shrinkage are not on the path)",
}


class _Optimizer:
    """Keras 2.5 ``optimizer_v2`` hyper-parameters.  ``learning_rate`` is a number or an instance of one of the
    four schedules of ``bore_b200.schedules``, which the kernels evaluate every step.  ``decay``, ``clipnorm``,
    ``clipvalue``, ``global_clipnorm`` and other callables as the learning rate are not taken: the kernels apply
    the plain rule."""

    kind = None

    def __init__(self, learning_rate, name, kwargs):
        if kwargs:
            raise TypeError(f"{type(self).__name__}: unsupported arguments {sorted(kwargs)} (decay, gradient "
                            "clipping and the like are not in the training kernels)")
        if type(learning_rate) in schedules.SCHEDULES:
            learning_rate.native()  # its arguments are refused here, not at the first fit
            self.learning_rate = learning_rate
        elif callable(learning_rate):
            raise NotImplementedError(
                f"{type(self).__name__}: the learning-rate schedules in the training kernels are "
                f"bore_b200.schedules.{{{', '.join(c.__name__ for c in schedules.SCHEDULES)}}}; another callable "
                f"(a function or a LearningRateSchedule subclass) runs Python, which the kernels cannot, got "
                f"{learning_rate!r}")
        else:
            self.learning_rate = float(learning_rate)
        self.name = name

    def hyper(self):
        """(BORE_OPT_* code, the BORE_OPT_NHP hyper-parameters of bore_mlp_set_optimizer_kind).  Under a schedule
        the learning-rate entry is 1, a stand-in the kernels do not read (lr_schedule gives the rate)."""
        g = lambda k: float(getattr(self, k, 0.0))  # noqa: E731
        rho = getattr(self, "rho", None)
        lr = 1.0 if isinstance(self.learning_rate, schedules.LearningRateSchedule) else self.learning_rate
        return OPT_CODES[self.kind], [lr, g("beta_1") if rho is None else float(rho), g("beta_2"),
                                      self.epsilon, g("momentum"), g("initial_accumulator_value"),
                                      float(bool(getattr(self, "centered", False)))]

    def lr_schedule(self):
        """(BORE_LR_* code, the parameters of bore_mlp_set_lr_schedule): BORE_LR_CONSTANT and none for a
        constant learning rate."""
        if isinstance(self.learning_rate, schedules.LearningRateSchedule):
            return self.learning_rate.native()
        return schedules.LR_CODES["constant"], []


class Adam(_Optimizer):
    """``keras.optimizers.Adam`` hyper-parameters (Keras defaults; epsilon is OUTSIDE the bias
    correction, unlike torch.optim.Adam)."""

    kind = "adam"

    def __init__(self, learning_rate=1e-3, beta_1=0.9, beta_2=0.999, epsilon=1e-7, amsgrad=False, name="Adam",
                 **kwargs):
        super().__init__(learning_rate, name, kwargs)
        if amsgrad:
            raise NotImplementedError("Adam(amsgrad=True) needs a third slot per parameter (vhat), which changes "
                                      "the shared-memory plan of every training kernel")
        self.beta_1, self.beta_2, self.epsilon = float(beta_1), float(beta_2), float(epsilon)
        self.amsgrad = False


class RMSprop(_Optimizer):
    """``keras.optimizers.RMSprop``: with momentum, epsilon is INSIDE the root (ResourceApplyRMSProp)."""

    kind = "rmsprop"

    def __init__(self, learning_rate=1e-3, rho=0.9, momentum=0.0, epsilon=1e-7, centered=False, name="RMSprop",
                 **kwargs):
        super().__init__(learning_rate, name, kwargs)
        self.rho, self.momentum, self.epsilon = float(rho), float(momentum), float(epsilon)
        self.centered = bool(centered)
        if self.centered and self.momentum > 0:
            raise NotImplementedError("RMSprop(centered=True, momentum>0) needs a third slot per parameter, which "
                                      "changes the shared-memory plan of every training kernel")


class Adagrad(_Optimizer):
    """``keras.optimizers.Adagrad``: the accumulator starts at ``initial_accumulator_value``."""

    kind = "adagrad"

    def __init__(self, learning_rate=1e-3, initial_accumulator_value=0.1, epsilon=1e-7, name="Adagrad", **kwargs):
        super().__init__(learning_rate, name, kwargs)
        self.initial_accumulator_value, self.epsilon = float(initial_accumulator_value), float(epsilon)


class Adadelta(_Optimizer):
    """``keras.optimizers.Adadelta``."""

    kind = "adadelta"

    def __init__(self, learning_rate=1e-3, rho=0.95, epsilon=1e-7, name="Adadelta", **kwargs):
        super().__init__(learning_rate, name, kwargs)
        self.rho, self.epsilon = float(rho), float(epsilon)


class Adamax(_Optimizer):
    """``keras.optimizers.Adamax``."""

    kind = "adamax"

    def __init__(self, learning_rate=1e-3, beta_1=0.9, beta_2=0.999, epsilon=1e-7, name="Adamax", **kwargs):
        super().__init__(learning_rate, name, kwargs)
        self.beta_1, self.beta_2, self.epsilon = float(beta_1), float(beta_2), float(epsilon)


class Nadam(_Optimizer):
    """``keras.optimizers.Nadam`` (its learning rate is not decayed; the momentum cache is per model).  A
    learning-rate schedule is a ValueError, as in Keras 2.5."""

    kind = "nadam"

    def __init__(self, learning_rate=1e-3, beta_1=0.9, beta_2=0.999, epsilon=1e-7, name="Nadam", **kwargs):
        if isinstance(learning_rate, schedules.LearningRateSchedule):
            raise ValueError("The Nadam optimizer does not support tf.keras.optimizers.LearningRateSchedules as "
                             "the learning rate.")
        super().__init__(learning_rate, name, kwargs)
        self.beta_1, self.beta_2, self.epsilon = float(beta_1), float(beta_2), float(epsilon)


_OPT_CLASSES = {c.kind: c for c in (Adam, RMSprop, Adagrad, Adadelta, Adamax, Nadam)}


def optimizer_spec(optimizer, owner="compile"):
    """The optimizer object for ``optimizer``: a Keras name (case-insensitive, as ``keras.optimizers.get``
    takes it), which gets the Keras defaults, or an instance of one of the classes above.  Optimizers
    without a kernel raise NotImplementedError saying why, unknown names ValueError."""
    if isinstance(optimizer, str):
        key = optimizer.lower()
        if key in _OPT_REFUSED:
            raise NotImplementedError(f"{owner}: optimizer {optimizer!r}: {_OPT_REFUSED[key]}")
        if key not in _OPT_CLASSES:
            raise ValueError(f"{owner}: optimizer must be one of {tuple(OPT_CODES)}, got {optimizer!r}")
        return _OPT_CLASSES[key]()
    if isinstance(optimizer, _Optimizer):
        return optimizer
    raise NotImplementedError(f"{owner}: optimizer must be a name in {tuple(OPT_CODES)} or one of "
                              f"bore_b200.layers.{{Adam, RMSprop, Adagrad, Adadelta, Adamax, Nadam}}, "
                              f"got {optimizer!r}")
