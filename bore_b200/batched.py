"""Batched BO problems (build extension; BASELINE.json configs[3]).

The reference runs ONE problem per Python process: ``classifier.fit(X, z)`` then
``classifier.argmax(...)`` (README.rst:83-103).  ``BatchedMaximizableSequential`` holds M
independent classifiers of one architecture -- seeds of a benchmark, concurrent optimisations,
per-budget classifiers -- and advances all of them with the same kernels in the same launches:
training is one CTA per model (``bore_mlp_fit``), screening / top-k / selection are grouped by
model, and the L-BFGS-B stepper sees M * num_starts starts.  Per problem the semantics are the
reference's own ``fit`` and ``argmax`` (bore/mixins.py:22-89); problems share nothing, so sharding
them over GPUs (``problem_shard``) needs no collective.
"""
import numpy as np
from scipy.optimize import OptimizeResult
from sklearn.utils import check_random_state

from . import ops
from .engine import NativeMLP, lbfgsb_message
from .layers import Dense, BinaryCrossentropy, optimizer_spec
from .models import check_class_weight, sample_weights
from .optimizers.utils import from_bounds
from .ragged import ragged_inputs, ragged_rows


def problem_shard(n_problems, rank, world):
    """Contiguous block [lo, hi) of problems owned by ``rank`` (no data-path collective)."""
    from .distributed import shard_bounds
    return shard_bounds(n_problems, rank, world)


class LazyLoss:
    """The (M, epochs) epoch losses of a batched ``fit``, fetched from the device the first time
    they are looked at: the training kernel is launched asynchronously, so the host is free to
    stage the next ``argmax``'s screening samples while the GPU trains (the single-model
    ``History`` of ``models.py`` does the same).  Behaves like the ndarray it wraps."""

    def __init__(self, loss_dev, layout=None):
        self._dev, self._host, self._layout = loss_dev, None, layout
        if layout is None:
            self.shape = tuple(loss_dev.shape)
        else:  # ragged problems: the losses come concatenated, problem p has layout.epochs[p] of them
            self.shape = (len(layout), int(layout.epochs.max()))
            self.epochs = layout.epochs.copy()

    def numpy(self):
        if self._host is None:
            self._host = self._dev.cpu().numpy()
            if self._layout is not None:
                self._host = self._layout.pad_loss(self._host)
            self._dev = None
        return self._host

    def first_last(self):
        """Every problem's first and last epoch loss (NaN for a problem that did not train)."""
        a = self.numpy()
        if a.shape[1] == 0:
            return np.full(a.shape[0], np.nan), np.full(a.shape[0], np.nan)
        if self._layout is None:
            return a[:, 0], a[:, -1]
        last = np.maximum(self._layout.epochs - 1, 0)
        return a[:, 0], a[np.arange(a.shape[0]), last]

    def __array__(self, dtype=None, copy=None):
        a = self.numpy()
        return a if dtype is None else a.astype(dtype)

    def __getitem__(self, idx):
        return self.numpy()[idx]

    def __len__(self):
        return self.shape[0]

    def __iter__(self):
        return iter(self.numpy())

    def __repr__(self):
        return repr(self.numpy())


class BatchedResults:
    """One ``OptimizeResult`` (or None) per problem, as a read-only sequence over the arrays that
    came back from the GPU: ``res[p]`` / iteration build the reference's per-problem objects on
    demand (4,096 of them cost more host time than the transfer), the bulk views ``found``, ``x``,
    ``fun``, ``nit``, ``nfev``, ``status`` serve callers that want all problems at once."""

    def __init__(self, rec, dim):
        self._rec, self._dim = rec, dim
        self.found = rec[:, dim + 5] != 0              # False: no start of the problem qualified
        self.x = rec[:, :dim]
        self.fun = rec[:, dim].astype(np.float32)
        self.nit = rec[:, dim + 1].astype(np.int64)
        self.nfev = rec[:, dim + 2].astype(np.int64)
        self.status = rec[:, dim + 3].astype(np.int64)
        self._task = rec[:, dim + 4].astype(np.int64)

    def __len__(self):
        return self._rec.shape[0]

    def __getitem__(self, p):
        if isinstance(p, slice):
            return [self[i] for i in range(*p.indices(len(self)))]
        if p < 0:
            p += len(self)
        if not 0 <= p < len(self):
            raise IndexError(p)
        if not self.found[p]:
            return None
        st, nfev = int(self.status[p]), int(self.nfev[p])
        return OptimizeResult(x=self.x[p].copy(), fun=self.fun[p], nit=int(self.nit[p]), nfev=nfev, njev=nfev,
                              status=st, success=bool(st == 0), message=lbfgsb_message(st, int(self._task[p])))

    def __iter__(self):
        return (self[p] for p in range(len(self)))


class BatchedMaximizableSequential:

    def __init__(self, layers, n_problems, transform=ops.identity, seed=None, device=None):
        self.layers = list(layers)
        assert self.layers and all(isinstance(l, Dense) for l in self.layers)
        assert self.layers[0].input_dim is not None, "the first Dense layer needs input_dim"
        self.n_problems = int(n_problems)
        dims = [self.layers[0].input_dim] + [l.units for l in self.layers]
        acts = [l.activation for l in self.layers]
        self.dims, self.acts = dims, acts
        e = transform(-ops.Expr(self, (1,), (1,)))
        if not isinstance(e, ops.Expr) or e.sign != -1:
            raise NotImplementedError("transform must be one of bore_b200.ops.identity/sigmoid/exp")
        self._transform = e.transform
        self._net = NativeMLP(dims, acts, n_models=self.n_problems, device=device)
        self._rs = np.random.RandomState(seed)
        self._compiled = False
        for p in range(self.n_problems):  # glorot_uniform kernels, zero biases, per problem
            ws = []
            for fi, fo in zip(dims[:-1], dims[1:]):
                lim = np.sqrt(6.0 / (fi + fo))
                ws += [self._rs.uniform(-lim, lim, size=(fi, fo)).astype(np.float32),
                       np.zeros(fo, np.float32)]
            self._net.set_weights(ws, model=p)
        self._last_stats = {}

    # ------------------------------------------------------------------ keras-shaped surface
    def compile(self, optimizer="adam", loss="binary_crossentropy", metrics=None):
        optimizer = optimizer_spec(optimizer)
        final = self.acts[-1]
        from_logits = isinstance(loss, BinaryCrossentropy) and loss.from_logits
        if not (isinstance(loss, BinaryCrossentropy) or loss == "binary_crossentropy"):
            raise NotImplementedError("only binary cross-entropy is on the BORE path")
        if from_logits != (final == "linear"):
            raise NotImplementedError("sigmoid output + 'binary_crossentropy', or linear output + "
                                      "BinaryCrossentropy(from_logits=True)")
        self._net.set_optimizer_kind(optimizer)
        l2 = []
        for lyr in self.layers:
            for r in (lyr.kernel_regularizer, lyr.bias_regularizer):
                l2.append(0.0 if r is None else float(r.l2))
        self._net.set_regularizers(l2)
        self._compiled = True

    def set_weights(self, weights_per_problem):
        assert len(weights_per_problem) == self.n_problems
        for p, ws in enumerate(weights_per_problem):
            self._net.set_weights(ws, model=p)

    def get_weights(self):
        return [self._net.get_weights(model=p) for p in range(self.n_problems)]

    def fit(self, x, y, batch_size=32, epochs=1, permutations=None, shuffle=True, verbose=0,
            gamma=None, sample_weight=None, class_weight=None):
        """x (M, N, D), y (M, N): every problem trains on its own N observations, all in one
        launch.  ``permutations``: (epochs, N) shared by all problems or (M, epochs, N).
        Ragged problems: ``x`` a list of M arrays (N_p, D) and ``y`` of M arrays (N_p,); then
        ``epochs`` is an int or M ints (0 leaves a problem untouched), ``sample_weight`` and
        ``permutations`` are lists of M arrays (N_p,) and (epochs_p, N_p), and the loss has shape
        (M, max epochs_p), NaN beyond each problem's epochs (``LazyLoss.epochs``).  Per problem the
        result is that of a fit of the problem alone.
        With ``gamma`` given, ``y`` holds the RAW targets and every problem is labelled
        ``z = y < quantile(y, gamma)`` on the device (bore/data.py:31-35) before training.
        ``sample_weight`` (M, N), or (N,) shared by all problems, and ``class_weight``
        {0: w0, 1: w1} weight each sample's loss as Keras' ``fit`` does; with ``gamma`` the
        class weights are applied on the device to the labels made there.
        Returns the per-problem history loss, shape (M, epochs), as a ``LazyLoss`` (array-like;
        the launch is asynchronous and the values are fetched on first use)."""
        if not self._compiled:
            raise RuntimeError("You must compile your model before training/testing.")
        if isinstance(x, (list, tuple)):
            return self._fit_ragged(x, y, batch_size, epochs, permutations, shuffle, verbose, gamma,
                                    sample_weight, class_weight)
        X = np.asarray(x)
        z = np.asarray(y)
        M, N, D = X.shape
        assert M == self.n_problems and z.shape == (M, N) and D == self.dims[0]
        w = None
        if sample_weight is not None:
            sw = np.asarray(sample_weight, np.float32)
            if sw.shape not in ((M, N), (N,)):
                raise ValueError(f"sample_weight must have shape ({M}, {N}) or ({N},), got {sw.shape}")
            w = np.broadcast_to(sw, (M, N)).reshape(-1)
        w, cw = self._class_weights(class_weight, gamma, z.reshape(-1), w)
        z_dev = None
        if gamma is not None:
            z_dev = self._net.quantile_labels_dev(
                self._net.to_device(np.ascontiguousarray(z, np.float64), np.float64), gamma).reshape(-1)
        if permutations is None:
            if shuffle:
                permutations = np.stack([np.stack([self._rs.permutation(N) for _ in range(epochs)])
                                         for _ in range(M)])
            else:
                permutations = np.tile(np.arange(N), (epochs, 1))
        perm = np.ascontiguousarray(permutations, np.int32)
        shared_perm = perm.ndim == 2
        assert perm.shape == ((epochs, N) if shared_perm else (M, epochs, N))
        net = self._net
        loss = net.fit_dev(net.to_device(X.reshape(M * N, D), np.float32),
                           z_dev if z_dev is not None else
                           net.to_device(z.reshape(-1), np.float32),
                           N, int(batch_size), int(epochs), net.to_device(perm, np.int32),
                           model0=0, count=M, shared_data=False, shared_perm=shared_perm,
                           w_dev=None if w is None else net.to_device(w, np.float32), class_weight=cw)
        out = LazyLoss(loss)
        if verbose:
            print(f"fit: {M} problems x {epochs} epochs, mean loss {out[:, 0].mean():.4f} -> "
                  f"{out[:, -1].mean():.4f}")
        return out

    def _class_weights(self, class_weight, gamma, z, w):
        """(sample weights with Keras' class weights folded in, class weights for labels made on the
        device): the rule of ``fit`` for host labels ``z`` or, with ``gamma``, device labels."""
        if class_weight is None:
            return w, None
        if gamma is None:  # labels known here: Keras' rule, class int(y)
            return sample_weights(z, w, class_weight), None
        cwd = check_class_weight(class_weight)  # labels 0 / 1 made on the device: both need a weight
        if not {0, 1} <= set(cwd):
            raise ValueError("class_weight needs weights for the classes 0 and 1 of the labels")
        return w, (cwd[0], cwd[1])

    def _fit_ragged(self, x, y, batch_size, epochs, permutations, shuffle, verbose, gamma, sample_weight,
                    class_weight):
        """``fit`` for lists of per-problem arrays (bore_mlp_fit_ragged): see ``fit``."""
        M, net = self.n_problems, self._net
        layout, X, z, w, perm = ragged_inputs(x, y, M, self.dims[0], epochs, sample_weight, permutations,
                                              self._rs, shuffle)
        w, cw = self._class_weights(class_weight, gamma, z, w)
        if gamma is not None:
            z_dev = net.quantile_labels_ragged_dev(net.to_device(z, np.float64), layout.n, gamma)
        else:
            z_dev = net.to_device(z, np.float32)
        loss = net.fit_ragged_dev(net.to_device(X, np.float32), z_dev, layout, int(batch_size),
                                  net.to_device(perm, np.int32), model0=0,
                                  w_dev=None if w is None else net.to_device(w, np.float32), class_weight=cw)
        out = LazyLoss(loss, layout)
        if verbose:
            first, last = out.first_last()
            trained = layout.epochs > 0
            msg = (f"mean loss {first[trained].mean():.4f} -> {last[trained].mean():.4f}" if trained.any()
                   else "nothing trained")
            print(f"fit: {M} problems x {layout.epochs.min()}..{layout.epochs.max()} epochs, {msg}")
        return out

    def predict(self, x):
        X = np.asarray(x)
        M, P, D = X.shape
        assert M == self.n_problems
        out = self._net.predict_multi_dev(self._net.to_device(X, np.float32))
        return out.cpu().numpy().reshape(M, P, 1)

    # ------------------------------------------------------------------ argmax per problem
    def argmax(self, bounds, num_starts=5, num_samples=1024, method="L-BFGS-B",
               options=dict(maxiter=1000, ftol=1e-9), random_state=None, X_init=None,
               exclude=None, rtol=1e-5, atol=1e-8, distortion=None):
        """One ``OptimizeResult`` (or None) per problem (``BatchedResults``, a lazy sequence):
        bore/mixins.py:22-89 for each of them.
        ``random_state`` draws the (M, num_samples, D) screening samples problem after problem
        (what M sequential ``argmax`` calls sharing one RandomState would consume); ``X_init``
        overrides the draw.  ``exclude`` (M, N, D), or a list of M arrays (n_p, D) with n_p >= 0: each
        problem's stored observations -- results
        ``np.allclose`` to one of them are dropped before the selection, which is the plugin's
        ``filter_fn=_is_unique`` (bore/plugins/hpbandster/base.py:227-231, bore/data.py:42-48).
        ``distortion``: the plugin's truncated-normal resample of the suggestion
        (``maybe_distort``, bore/base.py:45-64; plugins/hpbandster/base.py:266) applied to every
        problem's winner on the device; the uniform variates come from ``random_state`` AFTER the
        screening samples, one row per problem (problems without a winner consume theirs too)."""
        import torch
        assert num_samples >= num_starts > 0
        if isinstance(exclude, (list, tuple)):  # ragged: checked before anything is drawn or enqueued
            n_prev, prev = ragged_rows(exclude, self.n_problems, self.dims[0])
        if method != "L-BFGS-B":
            raise NotImplementedError("only L-BFGS-B has a device path")
        (low, high), dim = from_bounds(bounds)
        low, high = np.asarray(low, np.float64), np.asarray(high, np.float64)
        assert dim == self.dims[0]
        M, net = self.n_problems, self._net
        if X_init is None:
            # the reference's draw, problem after problem, from the caller's generator (same stream, same state
            # afterwards: bore_b200/hostrng.py), straight into the pinned staging buffer of the upload
            rs = check_random_state(random_state)
            X64, _ = net.uniform_to_device(rs, low, high, M * num_samples, dim)
            X64 = X64.view(M, num_samples, dim)
        else:
            rs = check_random_state(random_state) if distortion is not None else None
            X_init = np.asarray(X_init, np.float64)
            assert X_init.shape == (M, num_samples, dim)
            X64 = net.to_device(X_init, np.float64)
        z_init = net.predict_multi_dev(X64.to(torch.float32))
        if num_starts < num_samples:
            ind = net.topk_groups(z_init, num_starts, negate=True)     # (M, k) within-problem
            X0 = torch.gather(X64, 1, ind.to(torch.int64).unsqueeze(-1).expand(-1, -1, dim)).contiguous()
        else:
            X0 = X64
        opts = dict(options or {})
        res = net.lbfgsb_multi_dev(X0, low, high, transform=self._transform,
                                   m=opts.get("maxcor", 10), ftol=opts.get("ftol", 2.2204460492503131e-09),
                                   gtol=opts.get("gtol", 1e-5), maxiter=opts.get("maxiter", 15000),
                                   maxfun=opts.get("maxfun", 15000), maxls=opts.get("maxls", 20))
        keep = None
        if isinstance(exclude, (list, tuple)):  # ragged: problem p stores its own n_p rows
            keep = net.keep_unique_ragged_dev(res["x"], n_prev, net.to_device(prev, np.float64), rtol=rtol,
                                              atol=atol)
        elif exclude is not None:
            prev = np.ascontiguousarray(exclude, np.float64)
            assert prev.ndim == 3 and prev.shape[0] == M and prev.shape[2] == dim
            if prev.shape[1] > 0:
                keep = net.keep_unique_dev(res["x"], net.to_device(prev, np.float64), rtol=rtol, atol=atol)
        keys = net.select_best_groups(res["fun"], res["status"], keep_dev=keep)
        self._last_stats = dict(evals=res["evals"], rounds=res["rounds"], num_starts=num_starts)
        # one small record per problem leaves the GPU
        win = (0x7fffffff - (keys & 0x7fffffff)).clamp(0, num_starts - 1)
        pick = lambda t: torch.gather(t, 1, win.unsqueeze(-1)).squeeze(-1)
        xw = torch.gather(res["x"], 1, win.view(M, 1, 1).expand(-1, 1, dim)).squeeze(1)
        if distortion is not None:
            u = net.to_device(rs.uniform(size=(M, dim)), np.float64)
            xw = net.distort_dev(xw.contiguous(), distortion, low, high, u)
        rec = torch.cat([xw, pick(res["fun"]).unsqueeze(-1)] +
                        [pick(res[k]).to(torch.float64).unsqueeze(-1) for k in ("nit", "nfev", "status", "task")] +
                        [keys.to(torch.float64).unsqueeze(-1)], dim=1).cpu().numpy()
        return BatchedResults(rec, dim)
