"""Keras-shaped declarations the hot path needs: Dense, l2, BinaryCrossentropy and the optimizers.

Keras itself is absent (and not wanted on the path); these are plain spec objects that
``bore_b200.models.Sequential`` lowers onto the native handle.  Names and arguments follow
the call sites README.rst:60-66 and bore/plugins/hpbandster/base.py:113-116,147-158."""

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


class L2:
    """``keras.regularizers.l2(l2)``: adds ``l2 * sum(w**2)`` to the loss."""

    def __init__(self, l2=0.01):
        self.l2 = float(l2)


def l2(l2=0.01):
    return L2(l2)


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
        self.kernel_regularizer = kernel_regularizer
        self.bias_regularizer = bias_regularizer


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
    """Keras 2.5 ``optimizer_v2`` hyper-parameters.  ``decay``, ``clipnorm``, ``clipvalue``,
    ``global_clipnorm`` and learning-rate schedules are not taken: the kernels apply the plain rule."""

    kind = None

    def __init__(self, learning_rate, name, kwargs):
        if kwargs:
            raise TypeError(f"{type(self).__name__}: unsupported arguments {sorted(kwargs)} (decay, gradient "
                            "clipping and the like are not in the training kernels)")
        if callable(learning_rate):
            raise NotImplementedError(f"{type(self).__name__}: learning-rate schedules are not in the training "
                                      "kernels")
        self.learning_rate = float(learning_rate)
        self.name = name

    def hyper(self):
        """(BORE_OPT_* code, the BORE_OPT_NHP hyper-parameters of bore_mlp_set_optimizer_kind)."""
        g = lambda k: float(getattr(self, k, 0.0))  # noqa: E731
        rho = getattr(self, "rho", None)
        return OPT_CODES[self.kind], [self.learning_rate, g("beta_1") if rho is None else float(rho), g("beta_2"),
                                      self.epsilon, g("momentum"), g("initial_accumulator_value"),
                                      float(bool(getattr(self, "centered", False)))]


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
    """``keras.optimizers.Nadam`` (its learning rate is not decayed; the momentum cache is per model)."""

    kind = "nadam"

    def __init__(self, learning_rate=1e-3, beta_1=0.9, beta_2=0.999, epsilon=1e-7, name="Nadam", **kwargs):
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
