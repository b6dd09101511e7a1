"""Model surface (mirror of bore/models.py:9-33 plus the slice of keras.Sequential the hot path
uses: add / compile / fit / predict / evaluate / get_weights / set_weights / summary).

Keras cannot be subclassed here (absent, and TF must not be on the path), so ``Sequential`` is a
small container of ``Dense`` specs that lowers onto a native ``bore_mlp`` handle: training is the
fused CUDA fit kernel, inference the fused forward kernel.  Build-only extensions needed for
parity testing: ``fit(..., permutations=...)`` and ``get/set_optimizer_state``.

``StackedRecurrentFactory`` (the LSTM multi-fidelity classifier, bore/models.py:48-104) lives in
``bore_b200.recurrent`` and is re-exported here under the reference's module path.
"""
import numpy as np

from . import ops
from .layers import Dense, BinaryCrossentropy, optimizer_spec
from .mixins import MaximizableMixin, BatchMaximizableMixin


def check_class_weight(class_weight):
    """Keras' check of ``class_weight`` (data_adapter._make_class_weight_map_fn): the keys must be
    exactly the classes 0 .. K-1.  Returns {class: weight}."""
    keys = sorted(class_weight)
    if keys != list(range(len(keys))):
        raise ValueError(f"Expected `class_weight` to be a dict with keys from 0 to one less than the "
                         f"number of classes, found {class_weight}")
    return {int(k): float(v) for k, v in class_weight.items()}


def check_sample_weight(sample_weight, n):
    """``sample_weight`` of n samples, shape (n,) or (n, 1) -> float32 (n,); values pass unchecked."""
    w = np.asarray(sample_weight, np.float32)
    if w.shape not in ((n,), (n, 1)):
        raise ValueError(f"sample_weight must have shape ({n},) or ({n}, 1), got {w.shape}")
    return np.ascontiguousarray(w.reshape(n))


def sample_weights(z, sample_weight=None, class_weight=None):
    """Keras' weight of every sample of labels ``z`` (N,): ``sample_weight`` times the class weight of
    the sample's class int(z_i); None when neither is given.  A class without a key raises."""
    n = len(z)
    w = None if sample_weight is None else check_sample_weight(sample_weight, n)
    if class_weight is not None:
        cw = check_class_weight(class_weight)
        cls = np.asarray(z).reshape(n).astype(np.int64)
        missing = sorted(set(np.unique(cls).tolist()) - set(cw))
        if missing:
            raise ValueError(f"class_weight has no weight for the classes {missing} of the labels")
        by_class = np.array([cw[c] for c in range(len(cw))], np.float32)[cls]
        w = by_class if w is None else w * by_class
    return w


class History:
    """``history["loss"]`` like Keras' History.  ``loss`` may be a zero-argument callable: the
    training kernel is launched asynchronously and the epoch losses are fetched from the device
    the first time ``history`` is read, so ``fit`` does not stall the host."""

    def __init__(self, loss, epochs=None):
        self._loss = loss
        self._history = None
        self.epoch = list(range(len(loss) if epochs is None else epochs))

    @property
    def history(self):
        if self._history is None:
            loss = self._loss() if callable(self._loss) else self._loss
            self._history = {"loss": [float(v) for v in loss]}
            self._loss = None
        return self._history


class Sequential:
    """Stack of ``Dense`` layers with a scalar output."""

    def __init__(self, layers=None, seed=None, device=None):
        self.layers = []
        self._net = None
        self._rs = np.random.RandomState(seed)
        self._device = device
        self._compiled = None
        self._pending_weights = None
        for layer in layers or []:
            self.add(layer)

    # ------------------------------------------------------------------ construction
    def add(self, layer):
        if not isinstance(layer, Dense):
            raise NotImplementedError("only Dense layers are on the BORE-MLP path")
        if self._net is not None:
            raise RuntimeError("cannot add layers after the model was built")
        self.layers.append(layer)

    @property
    def input_dim(self):
        return self.layers[0].input_dim if self.layers else None

    def _l2(self):
        """Per-array l2 factors in Keras weight order [k0, b0, k1, b1, ...] (the plugin
        regularises its hidden layers only: plugins/hpbandster/base.py:113-116,152-155)."""
        out = []
        for lyr in self.layers:
            for r in (lyr.kernel_regularizer, lyr.bias_regularizer):
                out.append(0.0 if r is None else float(r.l2))
        return out

    def _engine(self, input_dim=None):
        """Build (once) the native handle; Keras builds lazily at the first call too."""
        if self._net is not None:
            if input_dim is not None and int(input_dim) != self._net.D:
                raise ValueError(f"expected input dimension {self._net.D}, got {input_dim}")
            return self._net
        if not self.layers:
            raise RuntimeError("the model has no layers")
        D = self.input_dim if self.input_dim is not None else input_dim
        if D is None:
            raise RuntimeError("input dimension unknown: pass input_dim to the first Dense layer "
                               "or call fit/predict first")
        from .engine import NativeMLP
        dims = [int(D)] + [lyr.units for lyr in self.layers]
        acts = [lyr.activation for lyr in self.layers]
        net = NativeMLP(dims, acts, n_models=1, device=self._device)
        if self._pending_weights is not None:
            net.set_weights(self._pending_weights)
            self._pending_weights = None
        else:
            ws = []
            for fi, fo in zip(dims[:-1], dims[1:]):  # glorot_uniform kernels, zero biases
                lim = np.sqrt(6.0 / (fi + fo))
                ws.append(self._rs.uniform(-lim, lim, size=(fi, fo)).astype(np.float32))
                ws.append(np.zeros(fo, np.float32))
            net.set_weights(ws)
        if self._compiled is not None:
            net.set_optimizer_kind(self._compiled["optimizer"])
        self._net = net
        return net

    def compile(self, optimizer="adam", loss=None, metrics=None, **kwargs):
        optimizer = optimizer_spec(optimizer)
        final = self.layers[-1].activation if self.layers else None
        if isinstance(loss, str):
            if loss != "binary_crossentropy":
                raise NotImplementedError("only binary cross-entropy is on the BORE path")
            loss = BinaryCrossentropy(from_logits=False)
        if not isinstance(loss, BinaryCrossentropy):
            raise NotImplementedError("loss must be 'binary_crossentropy' or BinaryCrossentropy")
        if loss.from_logits and final != "linear":
            raise NotImplementedError("BinaryCrossentropy(from_logits=True) needs a linear output layer")
        if not loss.from_logits and final != "sigmoid":
            raise NotImplementedError("'binary_crossentropy' needs a sigmoid output layer "
                                      "(Keras then takes the loss on its logits)")
        self._compiled = dict(optimizer=optimizer, loss=loss, metrics=list(metrics or []))
        if self._net is not None:
            self._net.set_optimizer_kind(optimizer)

    # ------------------------------------------------------------------ weights
    def get_weights(self):
        if self._net is None and self._pending_weights is not None:
            return [np.array(w) for w in self._pending_weights]
        return self._engine().get_weights()

    def set_weights(self, weights):
        if self._net is None and self.input_dim is None:
            # infer the input dimension from W0 like Keras would have from a built model
            self.layers[0].input_dim = int(np.asarray(weights[0]).shape[0])
        self._engine().set_weights(weights)

    def get_optimizer_state(self):
        """(slot 0 list, slot 1 list, iterations) -- Adam's m and v, or the slots of the compiled optimizer
        (DESIGN.md, "Optimizers"), and under Nadam its momentum cache as a fourth entry.  Persists across
        fit() calls like in Keras."""
        return self._engine().get_optimizer_state()

    def set_optimizer_state(self, m, v, iterations, cache=None):
        self._engine().set_optimizer_state(m, v, iterations, cache)

    def count_params(self):
        dims = [self.input_dim] + [lyr.units for lyr in self.layers]
        return sum(a * b + b for a, b in zip(dims[:-1], dims[1:]))

    def summary(self, print_fn=print):
        print_fn('Model: "sequential" (bore_b200 native, sm_100a)')
        fi = self.input_dim
        for i, lyr in enumerate(self.layers):
            n = "?" if fi is None else fi * lyr.units + lyr.units
            print_fn(f"dense_{i} (Dense)  output=(None, {lyr.units})  activation={lyr.activation}  params={n}")
            fi = lyr.units
        if self.input_dim is not None:
            print_fn(f"Total params: {self.count_params()}")

    # ------------------------------------------------------------------ training / inference
    def fit(self, x, y, batch_size=None, epochs=1, verbose=1, callbacks=None, shuffle=True,
            permutations=None, sample_weight=None, class_weight=None, **kwargs):
        """Minibatch Adam on binary cross-entropy, the whole run in one kernel launch.
        Returns a ``History`` with ``history["loss"]`` (Keras' sample-weighted epoch means).

        ``sample_weight`` (N,) or (N, 1) and ``class_weight`` {0: w0, 1: w1} weight each sample's
        loss as Keras does: a minibatch's loss is sum(w_i bce_i) / batch size.

        ``permutations`` (epochs, N): explicit per-epoch shuffles (build extension for parity);
        otherwise drawn from the model's RandomState when ``shuffle`` else the identity."""
        if kwargs:
            raise TypeError(f"fit: unsupported arguments {sorted(kwargs)}")
        if callbacks:
            raise NotImplementedError("callbacks cannot run inside the fused training kernel")
        if self._compiled is None:
            raise RuntimeError("You must compile your model before training/testing.")
        X = np.asarray(x)
        z = np.asarray(y).reshape(-1)
        N = X.shape[0]
        assert z.shape[0] == N, "x and y sizes do not match"
        w = sample_weights(z, sample_weight, class_weight)
        batch_size = 32 if batch_size is None else int(batch_size)
        epochs = int(epochs)
        net = self._engine(X.shape[1])
        if epochs <= 0 or N == 0:
            return History([])
        if permutations is None:
            if shuffle:
                permutations = np.stack([self._rs.permutation(N) for _ in range(epochs)])
            else:
                permutations = np.tile(np.arange(N), (epochs, 1))
        loss_dev = net.fit_async(X, z, epochs, batch_size, permutations, l2=self._l2(), w=w)
        hist = History(lambda: loss_dev.cpu().numpy()[0], epochs)
        if verbose:
            loss = hist.history["loss"]
            print(f"fit: {epochs} epochs x {-(-N // batch_size)} steps, "
                  f"loss {loss[0]:.4f} -> {loss[-1]:.4f}")
        return hist

    def predict(self, x, **kwargs):
        X = np.asarray(x)
        return self._engine(X.shape[1]).predict(X)

    def evaluate(self, x, y, verbose=0, sample_weight=None, **kwargs):
        """[loss, accuracy] (or the loss alone without metrics); ``sample_weight`` (N,) or (N, 1):
        loss sum(w_i bce_i) / N, accuracy sum(w_i hit_i) / sum(w_i) (0 when the weights sum to 0)."""
        if self._compiled is None:
            raise RuntimeError("You must compile your model before training/testing.")
        X = np.asarray(x)
        z = np.asarray(y).reshape(-1)
        w = sample_weights(z, sample_weight)
        out = self._engine(X.shape[1]).evaluate(X, z, l2=self._l2(), w=w)
        return out if self._compiled["metrics"] else out[0]

    def __call__(self, x):
        if isinstance(x, ops.Tracer):
            return ops.Expr(self, x.shape, tuple(x.shape[:-1]) + (1,))
        return self.predict(np.atleast_2d(np.asarray(x)))

    def _native_value_and_grad(self, X, transform, negate):
        return self._engine(X.shape[1]).value_and_grad(X, transform, negate)

    def _native_svgd(self, x_init, transform_fn, low, high, n_iter, opts):
        """SVGD on ``transform_fn(model(x))`` (maximised) with the whole loop on the device."""
        e = transform_fn(ops.Expr(self, (1,), (1,)))
        if not isinstance(e, ops.Expr) or e.sign != 1:
            raise NotImplementedError("transform must be one of bore_b200.ops.identity/sigmoid/exp")
        return self._engine(x_init.shape[-1]).svgd_maximize(x_init, e.transform, low, high, n_iter, **opts)


Model = Sequential


class DenseSequential(Sequential):
    """``num_layers`` hidden Dense layers + an output layer (bore/models.py:9-21).

    The reference's loop adds the first hidden layer TWICE (the ``if not i`` branch has no
    ``else``), so ``num_layers=2`` builds three hidden layers.  Reproduced on purpose: the plugin
    and the reference's own test go through this class."""

    def __init__(self, input_dim, output_dim, num_layers, num_units, layer_kws={},
                 final_layer_kws={}, **kwargs):
        super(DenseSequential, self).__init__(**kwargs)
        for i in range(num_layers):
            if not i:
                self.add(Dense(num_units, input_dim=input_dim, **layer_kws))
            self.add(Dense(num_units, **layer_kws))
        self.add(Dense(output_dim, **final_layer_kws))


class MaximizableModel(MaximizableMixin, Model):
    pass


class MaximizableSequential(MaximizableMixin, Sequential):
    pass


class MaximizableDenseSequential(MaximizableMixin, DenseSequential):
    pass


class BatchMaximizableModel(BatchMaximizableMixin, Model):
    pass


class BatchMaximizableSequential(BatchMaximizableMixin, Sequential):
    pass


class BatchMaximizableDenseSequential(BatchMaximizableMixin, DenseSequential):
    pass


from .recurrent import StackedRecurrentFactory, LSTMCell  # noqa: E402,F401  (bore/models.py:48-104)
