"""The LSTM multi-fidelity classifier (mirror of bore/models.py:48-104, SURVEY.md section 8f row 4).

``StackedRecurrentFactory`` owns ``num_layers`` ``LSTMCell`` specs and one ``Dense(1)`` and builds two
networks over the SAME weights, as the reference does by sharing Keras cell objects:

* ``build_many_to_many(mask_value)`` -- Masking -> RNN(cell, return_sequences=True)... ->
  TimeDistributed(Dense): the network ``fit`` trains on padded sequences
  (bore/plugins/hpbandster/multi_fidelity.py:198-233);
* ``build_one_to_one(num_steps, transform)`` -- RepeatVector -> the same cells -> the same Dense on the
  last step, a ``MaximizableSequential`` in the reference: its ``argmax`` proposes the next
  configuration (multi_fidelity.py:262-278).

Keras is absent and must not be on the path: both networks are thin views of one native ``bore_lstm``
handle (csrc/lstm.cu).  Training is one kernel launch; the argmax is the on-device L-BFGS-B stepper
(``bore_lbfgsb_init/step``) fed by ``bore_lstm_value_and_grad`` round by round -- no SciPy, no CPU
fallback.
"""
import ctypes as C
import os

import numpy as np

from . import _lib, ops
from .engine import ACT_CODES, OPT_NADAM, TRANSFORM_CODES, NativeMLP, _np_ptr, _ptr, _torch
from .layers import BinaryCrossentropy, Dense, activation_name, optimizer_spec, regularizer_factors, regularizer_get
from .mixins import MaximizableMixin
from .models import History

MAX_DIM, MAX_UNITS, MAX_LAYERS, MAX_STEPS, MAX_BATCH = 32, 32, 4, 8, 64  # csrc/lstm.cu limits


class LSTMCell:
    """``keras.layers.LSTMCell(units, activation="tanh", kernel_regularizer=None,
    recurrent_regularizer=None, bias_regularizer=None)``: gates i, f, c, o; sigmoid recurrent
    activation; glorot-uniform kernel, orthogonal recurrent kernel, zero bias with unit forget bias."""

    def __init__(self, units, activation="tanh", kernel_regularizer=None, recurrent_regularizer=None,
                 bias_regularizer=None, **kwargs):
        if kwargs:
            raise TypeError(f"LSTMCell: unsupported arguments {sorted(kwargs)}")
        activation = activation_name(activation, "LSTMCell")
        self.units = int(units)
        self.activation = activation
        self.kernel_regularizer = regularizer_get(kernel_regularizer, "LSTMCell")
        self.recurrent_regularizer = regularizer_get(recurrent_regularizer, "LSTMCell")
        self.bias_regularizer = regularizer_get(bias_regularizer, "LSTMCell")


class NativeLSTM:
    """Host-side owner of one ``bore_lstm*`` handle: moves buffers, nothing else."""

    # buffer plumbing shared with the MLP engine (it only needs .device / .lib)
    _tdev = NativeMLP._tdev
    _stream = NativeMLP._stream
    _staging = NativeMLP._staging
    to_device = NativeMLP.to_device
    uniform_to_device = NativeMLP.uniform_to_device
    topk_smallest = NativeMLP.topk_smallest
    select_best = NativeMLP.select_best
    keep_unique_dev = NativeMLP.keep_unique_dev

    def __init__(self, input_dim, units, num_layers, activation, device=None):
        self.lib = _lib.require_cuda()
        torch = _torch()
        if not torch.cuda.is_available():
            raise _lib.BoreNativeError("torch sees no CUDA device; bore_b200 has no CPU fallback")
        self.device = torch.cuda.current_device() if device is None else int(device)
        self.D, self.U, self.L = int(input_dim), int(units), int(num_layers)
        self.activation = "linear" if activation is None else activation
        h = C.c_void_p()
        _lib.check(self.lib.bore_lstm_create(self.D, self.U, self.L, ACT_CODES[self.activation],
                                             self.device, C.byref(h)))
        self.h = h
        self._pid = os.getpid()
        self.n_params = self.lib.bore_lstm_num_params(h)

    def __del__(self):
        h, self.h = getattr(self, "h", None), None
        if h and getattr(self, "_pid", None) == os.getpid():  # (a forked child must not touch CUDA)
            try:
                self.lib.bore_lstm_destroy(h)
            except Exception:
                pass

    # ------------------------------------------------------------------ parameters
    def shapes(self):
        """Keras ``get_weights()`` order: [K_l (in, 4U), R_l (U, 4U), b_l (4U)] per cell, then the
        Dense kernel (U, 1) and bias (1,)."""
        out, fan_in = [], self.D
        for _ in range(self.L):
            out += [(fan_in, 4 * self.U), (self.U, 4 * self.U), (4 * self.U,)]
            fan_in = self.U
        return out + [(self.U, 1), (1,)]

    _flatten = NativeMLP._flatten
    _unflatten = NativeMLP._unflatten

    def set_weights(self, weights):
        _lib.check(self.lib.bore_lstm_set_weights(self.h, _np_ptr(self._flatten(weights))))

    def get_weights(self):
        flat = np.empty(self.n_params, np.float32)
        _lib.check(self.lib.bore_lstm_get_weights(self.h, _np_ptr(flat)))
        return self._unflatten(flat)

    def set_adam_state(self, m, v, iterations):
        _lib.check(self.lib.bore_lstm_set_adam_state(self.h, _np_ptr(self._flatten(m)),
                                                     _np_ptr(self._flatten(v)), int(iterations)))

    def get_adam_state(self):
        mf, vf = np.empty(self.n_params, np.float32), np.empty(self.n_params, np.float32)
        it = C.c_int64()
        _lib.check(self.lib.bore_lstm_get_adam_state(self.h, _np_ptr(mf), _np_ptr(vf), C.byref(it)))
        return self._unflatten(mf), self._unflatten(vf), it.value

    opt_kind = 0  # BORE_OPT_* of the handle (Adam when created)

    def set_optimizer_kind(self, optimizer):
        """The optimizer and learning-rate schedule: a ``bore_b200.layers`` optimizer.  A new kind resets the
        state; a schedule keeps it and continues from ``iterations``."""
        kind, hp = optimizer.hyper()
        _lib.check(self.lib.bore_lstm_set_optimizer_kind(self.h, kind, _np_ptr(np.asarray(hp, np.float32))))
        code, sp = optimizer.lr_schedule()
        sp = np.asarray(sp, np.float32)
        _lib.check(self.lib.bore_lstm_set_lr_schedule(self.h, code, _np_ptr(sp), sp.size))
        self.opt_kind = kind

    def get_optimizer_state(self):
        """(slot 0, slot 1, iterations), and Nadam's momentum cache as a fourth entry under Nadam."""
        state = self.get_adam_state()
        if self.opt_kind != OPT_NADAM:
            return state
        c = C.c_float()
        _lib.check(self.lib.bore_lstm_get_nadam_cache(self.h, C.byref(c)))
        return state + (c.value,)

    def set_optimizer_state(self, m, v, iterations, cache=None):
        self.set_adam_state(m, v, iterations)
        if cache is not None:
            _lib.check(self.lib.bore_lstm_set_nadam_cache(self.h, float(cache)))

    def set_regularizers(self, l2, l1=None):
        """Per-array l2 and l1 factors in Keras weight order (3 per cell + 2); ``l1=None`` is no l1 penalty."""
        n = 3 * self.L + 2
        v = np.ascontiguousarray([float(t) for t in l2], np.float32)
        v1 = np.zeros(n, np.float32) if l1 is None else np.ascontiguousarray([float(t) for t in l1], np.float32)
        assert v.shape == (n,) and v1.shape == (n,)
        _lib.check(self.lib.bore_lstm_set_regularizers(self.h, _np_ptr(v)))
        _lib.check(self.lib.bore_lstm_set_l1_regularizers(self.h, _np_ptr(v1)))

    # ------------------------------------------------------------------ inference
    def predict_sequences_dev(self, X_dev, mask_value=None):
        """X_dev (S, T, D) float32 -> logits (S, T); steps equal to ``mask_value`` are masked."""
        torch = _torch()
        S, T, D = X_dev.shape
        assert D == self.D and X_dev.dtype == torch.float32 and X_dev.is_contiguous()
        out = torch.empty(S, T, dtype=torch.float32, device=self._tdev())
        _lib.check(self.lib.bore_lstm_predict_sequences(
            self.h, _ptr(X_dev), int(S), int(T), float(0.0 if mask_value is None else mask_value),
            0 if mask_value is None else 1, _ptr(out), self._stream()))
        return out

    def predict_steps_dev(self, X_dev, num_steps):
        """The one-to-one network: X_dev (S, D) float32 -> (S,) logits of step ``num_steps``."""
        torch = _torch()
        S, D = X_dev.shape
        assert D == self.D and X_dev.dtype == torch.float32 and X_dev.is_contiguous()
        out = torch.empty(S, dtype=torch.float32, device=self._tdev())
        _lib.check(self.lib.bore_lstm_predict(self.h, _ptr(X_dev), int(S), int(num_steps), _ptr(out),
                                              self._stream()))
        return out

    def value_and_grad_dev(self, X_dev, num_steps, transform="identity", negate=True, flags_dev=None,
                           f_dev=None, g_dev=None):
        """f = T(+-u(x)), g = df/dx of the one-to-one network; X_dev (S, D) float32 or float64."""
        torch = _torch()
        S, D = X_dev.shape
        assert D == self.D and X_dev.is_contiguous() and X_dev.dtype in (torch.float32, torch.float64)
        if f_dev is None:
            f_dev = torch.empty(S, dtype=torch.float32, device=self._tdev())
        if g_dev is None:
            g_dev = torch.empty(S, D, dtype=torch.float32, device=self._tdev())
        _lib.check(self.lib.bore_lstm_value_and_grad(
            self.h, int(num_steps), TRANSFORM_CODES[transform], 1 if negate else 0, _ptr(X_dev),
            1 if X_dev.dtype == torch.float64 else 0, int(S), _ptr(flags_dev), _ptr(f_dev), _ptr(g_dev),
            self._stream()))
        return f_dev, g_dev

    # ------------------------------------------------------------------ argmax
    def lbfgsb_dev(self, X0_dev, lo, hi, num_steps, transform="identity", m=10, ftol=1e-9, gtol=1e-5,
                   maxiter=1000, maxfun=15000, maxls=20):
        """All rows of X0_dev (S, D) float64 minimised on the device: the L-BFGS-B stepper posts the
        trial points, ``bore_lstm_value_and_grad`` answers them, one round of both per iteration of
        this loop.  Same result dict as ``NativeMLP.lbfgsb_dev``."""
        torch = _torch()
        S, D = X0_dev.shape
        assert D == self.D and X0_dev.dtype == torch.float64 and X0_dev.is_contiguous()
        dev = self._tdev()
        lo = np.ascontiguousarray(np.broadcast_to(np.asarray(lo, np.float64), (D,)))
        hi = np.ascontiguousarray(np.broadcast_to(np.asarray(hi, np.float64), (D,)))
        nbytes = self.lib.bore_lbfgsb_workspace_bytes(S, D, int(m))
        work = torch.empty(int(nbytes), dtype=torch.uint8, device=dev)
        xreq = torch.empty(S, D, dtype=torch.float64, device=dev)
        pend = torch.empty(S, dtype=torch.int32, device=dev)
        stream = self._stream()
        _lib.check(self.lib.bore_lbfgsb_init(_ptr(X0_dev), S, D, _np_ptr(lo), _np_ptr(hi), int(m),
                                             float(ftol), float(gtol), int(maxiter), int(maxfun),
                                             int(maxls), _ptr(work), work.numel(), _ptr(xreq),
                                             _ptr(pend), self.device, stream))
        f = torch.zeros(S, dtype=torch.float32, device=dev)
        g = torch.zeros(S, D, dtype=torch.float32, device=dev)
        pending, rounds = C.c_int(S), 0
        while pending.value > 0:
            self.value_and_grad_dev(xreq, num_steps, transform, True, flags_dev=pend, f_dev=f, g_dev=g)
            _lib.check(self.lib.bore_lbfgsb_step(_ptr(f), _ptr(g), 0, S, D, _ptr(work), _ptr(xreq),
                                                 _ptr(pend), C.byref(pending), self.device, stream))
            rounds += 1
        x = torch.empty(S, D, dtype=torch.float64, device=dev)
        fun = torch.empty(S, dtype=torch.float64, device=dev)
        ints = torch.empty(4, S, dtype=torch.int32, device=dev)
        _lib.check(self.lib.bore_lbfgsb_results(S, D, _ptr(work), _ptr(x), _ptr(fun), _ptr(ints[0]),
                                                _ptr(ints[1]), _ptr(ints[2]), _ptr(ints[3]),
                                                self.device, stream))
        return dict(x=x, fun=fun, nit=ints[0], nfev=ints[1], status=ints[2], task=ints[3],
                    rounds=rounds, evals=int(ints[1].sum().item()))

    # ------------------------------------------------------------------ training
    def fit_async(self, X, Y, epochs, batch_size, permutations, mask_value):
        """Keras ``fit`` on padded sequences X (N, T, D), Y (N, T[, 1]) with explicit per-epoch
        permutations -> (epochs,) device tensor of epoch losses (the launch is asynchronous)."""
        torch = _torch()
        X = np.asarray(X)
        N, T, D = X.shape
        assert D == self.D
        Y = np.asarray(Y).reshape(N, T)
        perm = np.ascontiguousarray(permutations, np.int32).reshape(epochs, N)
        loss = torch.empty(epochs, dtype=torch.float32, device=self._tdev())
        Xd, Yd = self.to_device(X, np.float32), self.to_device(Y, np.float32)
        _lib.check(self.lib.bore_lstm_fit(self.h, _ptr(Xd), _ptr(Yd), int(N), int(T),
                                          float(np.float32(mask_value)), int(batch_size), int(epochs),
                                          _ptr(self.to_device(perm, np.int32)), _ptr(loss), self._stream()))
        return loss

    def evaluate(self, X, Y, mask_value):
        X = np.asarray(X)
        N, T, D = X.shape
        out = np.zeros(2, np.float32)
        Xd = self.to_device(X, np.float32)
        Yd = self.to_device(np.asarray(Y).reshape(N, T), np.float32)
        _lib.check(self.lib.bore_lstm_evaluate(self.h, _ptr(Xd), _ptr(Yd), int(N), int(T),
                                               float(np.float32(mask_value)), _np_ptr(out), self._stream()))
        return [float(out[0]), float(out[1])]


def _orthogonal(rs, rows, cols):
    """Keras ``Orthogonal`` initialiser's construction: QR of a (max, min) normal matrix, signs of
    R's diagonal folded into Q, transposed when rows < cols."""
    a = rs.normal(size=(max(rows, cols), min(rows, cols)))
    q, r = np.linalg.qr(a)
    q = q * np.sign(np.diag(r))
    return (q.T if rows < cols else q)[:rows, :cols]


class StackedRecurrentFactory:
    """bore/models.py:48-104: same constructor and builders.  ``seed`` / ``device`` are build
    extensions (initial weights from a ``RandomState``; which GPU)."""

    def __init__(self, input_dim, output_dim, num_layers=2, num_units=32, layer_kws={},
                 final_layer_kws={}, seed=None, device=None):
        self.input_dim = input_dim

        assert "return_sequences" not in layer_kws
        assert "activation" not in final_layer_kws
        if output_dim != 1:
            raise NotImplementedError("the recurrent classifier has one logit per step (output_dim=1)")
        if not (1 <= input_dim <= MAX_DIM and 1 <= num_units <= MAX_UNITS and 1 <= num_layers <= MAX_LAYERS):
            raise NotImplementedError(f"csrc/lstm.cu limits: input_dim <= {MAX_DIM}, num_units <= {MAX_UNITS}, "
                                      f"num_layers <= {MAX_LAYERS}")

        # stack of recurrent cells + the fully-connected final layer
        self.cells = [LSTMCell(num_units, **layer_kws) for _ in range(num_layers)]
        self.final_layer = Dense(output_dim, **final_layer_kws)
        self._rs = np.random.RandomState(seed)
        self._device = device
        self._net = None

    # the one native handle behind every network this factory builds
    def _engine(self):
        if self._net is None:
            cell = self.cells[0]
            net = NativeLSTM(self.input_dim, cell.units, len(self.cells), cell.activation, self._device)
            ws, fan_in, U = [], self.input_dim, cell.units
            for _ in self.cells:
                lim = np.sqrt(6.0 / (fan_in + 4 * U))
                ws.append(self._rs.uniform(-lim, lim, size=(fan_in, 4 * U)).astype(np.float32))
                ws.append(_orthogonal(self._rs, U, 4 * U).astype(np.float32))
                b = np.zeros(4 * U, np.float32)
                b[U:2 * U] = 1.0  # unit_forget_bias
                ws.append(b)
                fan_in = U
            lim = np.sqrt(6.0 / (U + 1))
            ws.append(self._rs.uniform(-lim, lim, size=(U, 1)).astype(np.float32))
            ws.append(np.zeros(1, np.float32))
            net.set_weights(ws)
            net.set_regularizers(*self._factors())
            self._net = net
        return self._net

    def _factors(self):
        """Per-array (l2, l1) factors in Keras weight order: kernel, recurrent kernel, bias of every cell, then
        the final Dense layer's kernel and bias."""
        regs = [r for c in self.cells for r in (c.kernel_regularizer, c.recurrent_regularizer, c.bias_regularizer)]
        return regularizer_factors(regs + [self.final_layer.kernel_regularizer, self.final_layer.bias_regularizer])

    def _l2(self):
        return self._factors()[0]

    def build_many_to_many(self, mask_value=1e+9):
        """Training network: masked many-to-many logits (bore/models.py:69-83)."""
        return RecurrentSequential(self, mask_value)

    def build_one_to_one(self, num_steps, transform=ops.identity):
        """Acquisition network for rung ``num_steps - 1`` (bore/models.py:85-104)."""
        if not 1 <= num_steps <= MAX_STEPS:
            raise NotImplementedError(f"csrc/lstm.cu limit: num_steps <= {MAX_STEPS}")
        return MaximizableRecurrent(transform, self, num_steps)


class RecurrentSequential:
    """The many-to-many network: the slice of ``keras.Sequential`` the plugin uses
    (compile / fit / evaluate / predict / summary / get_weights / set_weights)."""

    def __init__(self, factory, mask_value):
        self.factory, self.mask_value = factory, mask_value
        self._compiled = None
        self._rs = factory._rs

    def compile(self, optimizer="adam", loss=None, metrics=None, **kwargs):
        optimizer = optimizer_spec(optimizer)
        if not isinstance(loss, BinaryCrossentropy) or not loss.from_logits:
            raise NotImplementedError("the recurrent classifier trains on BinaryCrossentropy(from_logits=True)")
        self._compiled = dict(optimizer=optimizer, loss=loss, metrics=list(metrics or []))
        if self.factory._net is not None:
            self.factory._net.set_optimizer_kind(optimizer)

    def get_weights(self):
        return self.factory._engine().get_weights()

    def set_weights(self, weights):
        self.factory._engine().set_weights(weights)

    def get_optimizer_state(self):
        """(slot 0, slot 1, iterations) -- and Nadam's momentum cache under Nadam."""
        return self._optimized_engine().get_optimizer_state()

    def set_optimizer_state(self, m, v, iterations, cache=None):
        self._optimized_engine().set_optimizer_state(m, v, iterations, cache)

    # the handle, running the compiled optimizer
    def _optimized_engine(self):
        net = self.factory._engine()
        if self._compiled is not None:
            net.set_optimizer_kind(self._compiled["optimizer"])
        return net

    def count_params(self):
        return sum(int(np.prod(s)) for s in self.factory._engine().shapes())

    def summary(self, print_fn=print):
        f = self.factory
        print_fn('Model: "sequential" (bore_b200 native LSTM stack, sm_100a)')
        print_fn(f"masking (Masking)  mask_value={self.mask_value}")
        fan_in = f.input_dim
        for i, c in enumerate(f.cells):
            print_fn(f"rnn_{i} (RNN LSTMCell)  output=(None, None, {c.units})  activation={c.activation}  "
                     f"params={4 * c.units * (fan_in + c.units + 1)}")
            fan_in = c.units
        print_fn(f"time_distributed (Dense)  output=(None, None, 1)  params={fan_in + 1}")

    def fit(self, x, y, batch_size=None, epochs=1, verbose=1, callbacks=None, shuffle=True,
            permutations=None, **kwargs):
        """The compiled optimizer on the masked BCE-with-logits of padded sequences x (N, T, D), y (N, T, 1); one
        kernel launch.  ``permutations`` (epochs, N) as in ``Sequential.fit``."""
        if kwargs:
            raise TypeError(f"fit: unsupported arguments {sorted(kwargs)}")
        if callbacks:
            raise NotImplementedError("callbacks cannot run inside the fused training kernel")
        if self._compiled is None:
            raise RuntimeError("You must compile your model before training/testing.")
        X = np.asarray(x)
        N, T = X.shape[0], X.shape[1]
        if T > MAX_STEPS:
            raise NotImplementedError(f"csrc/lstm.cu limit: at most {MAX_STEPS} rungs")
        batch_size = 32 if batch_size is None else int(batch_size)
        if batch_size > MAX_BATCH:
            raise NotImplementedError(f"csrc/lstm.cu limit: batch_size <= {MAX_BATCH}")
        epochs = int(epochs)
        if epochs <= 0 or N == 0:
            return History([])
        net = self._optimized_engine()
        net.set_regularizers(*self.factory._factors())
        if permutations is None:
            permutations = (np.stack([self._rs.permutation(N) for _ in range(epochs)]) if shuffle
                            else np.tile(np.arange(N), (epochs, 1)))
        loss_dev = net.fit_async(X, y, epochs, batch_size, permutations, self.mask_value)
        hist = History(lambda: loss_dev.cpu().numpy(), epochs)
        if verbose:
            loss = hist.history["loss"]
            print(f"fit: {epochs} epochs x {-(-N // batch_size)} steps, loss {loss[0]:.4f} -> {loss[-1]:.4f}")
        return hist

    def evaluate(self, x, y, verbose=0, **kwargs):
        if self._compiled is None:
            raise RuntimeError("You must compile your model before training/testing.")
        net = self.factory._engine()
        net.set_regularizers(*self.factory._factors())
        out = net.evaluate(x, y, self.mask_value)
        return out if self._compiled["metrics"] else out[0]

    def predict(self, x, **kwargs):
        """(N, T, D) -> logits (N, T, 1)."""
        net = self.factory._engine()
        X = np.asarray(x)
        out = net.predict_sequences_dev(net.to_device(X, np.float32), np.float32(self.mask_value))
        return out.cpu().numpy()[..., None]


class _OneToOneEngine:
    """What ``MaximizableMixin`` asks of an engine, answered by the one-to-one view of a
    ``NativeLSTM`` with a fixed number of steps."""

    def __init__(self, net, num_steps):
        self.net, self.num_steps, self.D = net, num_steps, net.D

    def __getattr__(self, name):  # to_device / topk_smallest / select_best / keep_unique_dev ...
        return getattr(self.net, name)

    def predict_dev(self, X_dev):
        return self.net.predict_steps_dev(X_dev, self.num_steps)

    def lbfgsb_dev(self, X0_dev, lo, hi, **kw):
        return self.net.lbfgsb_dev(X0_dev, lo, hi, self.num_steps, **kw)


class _OneToOneNetwork:
    """RepeatVector(num_steps) -> cells -> Dense on the last step (bore/models.py:85-104)."""

    def __init__(self, factory, num_steps):
        self.factory, self.num_steps = factory, int(num_steps)
        self._view = None

    @property
    def input_dim(self):
        return self.factory.input_dim

    def _engine(self, input_dim=None):
        if input_dim is not None and int(input_dim) != self.factory.input_dim:
            raise ValueError(f"expected input dimension {self.factory.input_dim}, got {input_dim}")
        if self._view is None:
            self._view = _OneToOneEngine(self.factory._engine(), self.num_steps)
        return self._view

    def get_weights(self):
        return self.factory._engine().get_weights()

    def predict(self, x, **kwargs):
        """(S, D) -> logits (S, 1) of step ``num_steps``."""
        net = self.factory._engine()
        X = np.atleast_2d(np.asarray(x))
        if X.shape[0] == 0:
            return np.zeros((0, 1), np.float32)
        return net.predict_steps_dev(net.to_device(X, np.float32), self.num_steps).cpu().numpy().reshape(-1, 1)

    def __call__(self, x):
        if isinstance(x, ops.Tracer):
            return ops.Expr(self, x.shape, tuple(x.shape[:-1]) + (1,))
        return self.predict(x)

    def _native_value_and_grad(self, X, transform, negate):
        net = self.factory._engine()
        f, g = net.value_and_grad_dev(net.to_device(np.atleast_2d(X), np.float32), self.num_steps,
                                      transform, negate)
        return f.cpu().numpy(), g.cpu().numpy()


class MaximizableRecurrent(MaximizableMixin, _OneToOneNetwork):
    """``MaximizableSequential`` over the one-to-one recurrent network: ``maxima`` / ``argmax`` with
    the reference's signatures (bore/mixins.py:22-89)."""
