"""Keras-shaped declarations the hot path needs: Dense, l2, BinaryCrossentropy, Adam.

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


class Adam:
    """``keras.optimizers.Adam`` hyper-parameters (Keras defaults; epsilon is OUTSIDE the bias
    correction, unlike torch.optim.Adam)."""

    def __init__(self, learning_rate=1e-3, beta_1=0.9, beta_2=0.999, epsilon=1e-7):
        self.learning_rate, self.beta_1, self.beta_2, self.epsilon = \
            float(learning_rate), float(beta_1), float(beta_2), float(epsilon)
