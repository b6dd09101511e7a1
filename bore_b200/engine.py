"""Host-side owner of one native model handle (``bore_mlp*``) and its device buffers.

Everything numeric happens in libbore_b200.so (hand-written sm_100a kernels) through the C ABI
of include/bore_b200.h; this class only moves buffers.  PyTorch is used for exactly three things:
device memory (``torch.empty(..., device="cuda")``), pinned host staging buffers and the current
CUDA stream.  There is no CPU fallback -- construction fails without a CUDA device.
"""
import ctypes as C
import os

import numpy as np

from . import _lib

# BORE_ACT_* of include/bore_b200.h
ACT_CODES = {"linear": 0, None: 0, "relu": 1, "elu": 2, "sigmoid": 3, "tanh": 4, "selu": 5, "softplus": 6,
             "softsign": 7, "hard_sigmoid": 8, "exponential": 9}
TRANSFORM_CODES = {"identity": 0, "sigmoid": 1, "exp": 2}
OPT_NADAM = 5  # BORE_OPT_NADAM (layers.OPT_CODES): the kind with a momentum cache

# scipy.optimize L-BFGS-B task codes -> message (scipy/optimize/_lbfgsb_py.py:49-90)
_STATUS_MSG = {0: "CONVERGENCE", 1: "STOP", 2: "ABNORMAL"}
_TASK_MSG = {0: "", 401: "NORM OF PROJECTED GRADIENT <= PGTOL",
             402: "RELATIVE REDUCTION OF F <= FACTR*EPSMCH",
             502: "TOTAL NO. OF F,G EVALUATIONS EXCEEDS LIMIT",
             504: "TOTAL NO. OF ITERATIONS REACHED LIMIT"}


def lbfgsb_message(status, task):
    return _STATUS_MSG.get(int(status), "?") + ": " + _TASK_MSG.get(int(task), "")


def _torch():
    import torch
    return torch


def _ptr(t):
    return C.c_void_p(t.data_ptr()) if t is not None else None


def _np_ptr(a):
    return a.ctypes.data_as(C.c_void_p)


class NativeMLP:
    """M independent MLPs of one architecture living on one GPU."""

    def __init__(self, dims, acts, n_models=1, device=None):
        self.lib = _lib.require_cuda()
        torch = _torch()
        if not torch.cuda.is_available():
            raise _lib.BoreNativeError("torch sees no CUDA device; bore_b200 has no CPU fallback")
        self.device = torch.cuda.current_device() if device is None else int(device)
        self.dims = [int(d) for d in dims]
        self.acts = [a if a is not None else "linear" for a in acts]
        assert len(self.acts) == len(self.dims) - 1
        codes = [ACT_CODES[a] for a in self.acts]
        self.n_models = int(n_models)
        h = C.c_void_p()
        dims_c = (C.c_int * len(self.dims))(*self.dims)
        acts_c = (C.c_int * len(codes))(*codes)
        _lib.check(self.lib.bore_mlp_create(len(codes), dims_c, acts_c, self.n_models, self.device,
                                            C.byref(h)))
        self.h = h
        self._pid = os.getpid()
        self.n_params = self.lib.bore_mlp_num_params(h)
        self.D = self.dims[0]
        self._work = None  # cached L-BFGS-B workspace (torch uint8 tensor)

    def __del__(self):
        h, self.h = getattr(self, "h", None), None
        if h and getattr(self, "_pid", None) == os.getpid():  # (a forked child must not touch CUDA)
            try:
                self.lib.bore_mlp_destroy(h)
            except Exception:
                pass

    # ------------------------------------------------------------------ helpers
    def _tdev(self):
        return _torch().device("cuda", self.device)

    def _stream(self):
        return C.c_void_p(_torch().cuda.current_stream(self.device).cuda_stream)

    def shapes(self):
        out = []
        for fi, fo in zip(self.dims[:-1], self.dims[1:]):
            out += [(fi, fo), (fo,)]
        return out

    def _flatten(self, weights):
        shp = self.shapes()
        assert len(weights) == len(shp), f"expected {len(shp)} arrays, got {len(weights)}"
        parts = []
        for w, s in zip(weights, shp):
            w = np.asarray(w, np.float32)
            assert w.shape == s, f"weight shape {w.shape} != {s}"
            parts.append(w.ravel())
        return np.ascontiguousarray(np.concatenate(parts))

    def _unflatten(self, flat):
        out, o = [], 0
        for s in self.shapes():
            k = int(np.prod(s))
            out.append(flat[o:o + k].reshape(s).copy())
            o += k
        return out

    def _staging(self, nbytes):
        """A cached pinned staging buffer of at least ``nbytes`` whose last upload has completed:
        ``[uint8 tensor, event]`` (None if page-locked memory cannot be had)."""
        torch = _torch()
        pool = self.__dict__.setdefault("_pinned", [])
        best = None
        for ent in pool:
            # a buffer serves payloads of its own size class only (>= a quarter of its capacity):
            # a small upload must not occupy the staging buffer of a large one, whose next use
            # would then have to page-lock a fresh buffer (~100 ms for 256 MB)
            if (ent[0].numel() >= nbytes and ent[0].numel() <= max(4 * nbytes, 1 << 16) and ent[1].query()
                    and (best is None or ent[0].numel() < best[0].numel())):
                best = ent
        if best is None:
            cap = 1 << max(12, int(nbytes - 1).bit_length())
            try:
                buf = torch.empty(cap, dtype=torch.uint8, pin_memory=True)
            except RuntimeError:
                return None
            best = [buf, torch.cuda.Event()]
            pool.append(best)
            if len(pool) > 16:  # drop the oldest idle buffer
                for i, ent in enumerate(pool[:-1]):
                    if ent[1].query():
                        del pool[i]
                        break
        return best

    def to_device(self, a, dtype):
        """numpy -> device tensor through a cached pinned staging buffer (page-locking a fresh
        buffer per call costs more than the copy itself).  A buffer is reused once the event
        recorded behind its last host-to-device copy has completed.  A dtype change (the float64
        arrays of the reference's surface -> the kernels' float32) happens in the same pass that
        fills the staging buffer, not in a temporary of its own."""
        torch = _torch()
        a = np.asarray(a)
        dtype = np.dtype(dtype)
        tdt = torch.from_numpy(np.empty(0, dtype)).dtype
        nbytes = a.size * dtype.itemsize
        if nbytes == 0:
            return torch.empty(a.shape, dtype=tdt, device=self._tdev())
        best = self._staging(nbytes)
        if best is None:
            return torch.from_numpy(np.ascontiguousarray(a, dtype=dtype)).to(self._tdev())
        view = best[0][:nbytes].view(tdt).reshape(a.shape)
        if nbytes >= (1 << 22) and a.flags.writeable and a.dtype.kind in "fiub":
            view.copy_(torch.from_numpy(a))  # large arrays: torch converts / copies on all host cores
        else:
            np.copyto(view.numpy(), a, casting="unsafe")
        out = view.to(self._tdev(), non_blocking=True)
        best[1].record(torch.cuda.current_stream(self.device))
        return out

    def uniform_to_device(self, random_state, low, high, n, dim):
        """``random_state.uniform(low, high, size=(n, dim))`` (bore/mixins.py:49: the candidate points of an
        argmax, drawn on the host from the caller's generator) written straight into the pinned staging
        buffer of its upload -> ``(float64 device tensor, host view)``.  The host view is valid until the
        next upload of this size class; callers that keep rows copy them."""
        from . import hostrng
        torch = _torch()
        nbytes = n * dim * 8
        best = self._staging(nbytes) if nbytes else None
        if best is None:
            X = hostrng.uniform(random_state, low, high, n, dim)
            return self.to_device(X, np.float64), X
        view = best[0][:nbytes].view(torch.float64).reshape(n, dim)
        host = view.numpy()
        hostrng.uniform(random_state, low, high, n, dim, out=host)
        out = view.to(self._tdev(), non_blocking=True)
        best[1].record(torch.cuda.current_stream(self.device))
        return out, host

    # ------------------------------------------------------------------ parameters
    def set_weights(self, weights, model=0):
        flat = self._flatten(weights)
        _lib.check(self.lib.bore_mlp_set_weights(self.h, model, _np_ptr(flat)))

    def get_weights(self, model=0):
        flat = np.empty(self.n_params, np.float32)
        _lib.check(self.lib.bore_mlp_get_weights(self.h, model, _np_ptr(flat)))
        return self._unflatten(flat)

    def set_adam_state(self, m, v, iterations, model=0):
        mf, vf = self._flatten(m), self._flatten(v)
        _lib.check(self.lib.bore_mlp_set_adam_state(self.h, model, _np_ptr(mf), _np_ptr(vf),
                                                    int(iterations)))

    def get_adam_state(self, model=0):
        mf = np.empty(self.n_params, np.float32)
        vf = np.empty(self.n_params, np.float32)
        it = C.c_int64()
        _lib.check(self.lib.bore_mlp_get_adam_state(self.h, model, _np_ptr(mf), _np_ptr(vf),
                                                    C.byref(it)))
        return self._unflatten(mf), self._unflatten(vf), it.value

    def reset_optimizer(self, model0=0, count=None):
        """The optimizer state of models [model0, model0 + count) back to its initial values (zeros; Adagrad's
        accumulator at initial_accumulator_value, Nadam's cache at 1) on the current stream (asynchronous)."""
        count = self.n_models - model0 if count is None else count
        _lib.check(self.lib.bore_mlp_reset_optimizer(self.h, model0, count, self._stream()))

    opt_kind = 0  # BORE_OPT_* of the handle (Adam when created)

    def set_optimizer(self, lr=1e-3, beta1=0.9, beta2=0.999, eps=1e-7):
        _lib.check(self.lib.bore_mlp_set_optimizer(self.h, lr, beta1, beta2, eps))
        self.opt_kind = 0

    def set_optimizer_kind(self, optimizer):
        """Every model's optimizer: a ``bore_b200.layers`` optimizer.  A new kind resets every model's state."""
        kind, hp = optimizer.hyper()
        _lib.check(self.lib.bore_mlp_set_optimizer_kind(self.h, kind, _np_ptr(np.asarray(hp, np.float32))))
        self.opt_kind = kind

    def get_optimizer_state(self, model=0):
        """(slot 0, slot 1, iterations), and Nadam's momentum cache as a fourth entry under Nadam."""
        state = self.get_adam_state(model)
        if self.opt_kind != OPT_NADAM:
            return state
        c = C.c_float()
        _lib.check(self.lib.bore_mlp_get_nadam_cache(self.h, model, C.byref(c)))
        return state + (c.value,)

    def set_optimizer_state(self, m, v, iterations, cache=None, model=0):
        self.set_adam_state(m, v, iterations, model)
        if cache is not None:
            _lib.check(self.lib.bore_mlp_set_nadam_cache(self.h, model, float(cache)))

    def set_fit_mode(self, mode):
        """0 automatic, 1 one CTA per model, 2 one thread-block cluster per model."""
        _lib.check(self.lib.bore_mlp_set_fit_mode(self.h, int(mode)))

    def set_regularizers(self, l2):
        """``l2``: one factor for every kernel and bias, or a per-array sequence in Keras weight
        order [k0, b0, k1, b1, ...]."""
        L = len(self.acts)
        v = [float(l2)] * (2 * L) if np.isscalar(l2) else [float(t) for t in l2]
        assert len(v) == 2 * L
        lk = np.ascontiguousarray(v[0::2], np.float32)
        lb = np.ascontiguousarray(v[1::2], np.float32)
        _lib.check(self.lib.bore_mlp_set_regularizers(self.h, _np_ptr(lk), _np_ptr(lb)))

    def params_tensor(self):
        """The flat [n_models, n_params] parameter block as a torch view (for NCCL broadcast)."""
        torch = _torch()
        p = C.c_void_p()
        _lib.check(self.lib.bore_mlp_params_dev(self.h, C.byref(p)))
        n = self.n_models * self.n_params

        class _Holder:  # __cuda_array_interface__ view of native memory
            pass
        hd = _Holder()
        hd.__cuda_array_interface__ = dict(shape=(n,), typestr="<f4", data=(p.value, False),
                                           version=3)
        return torch.as_tensor(hd, device=self._tdev()).view(self.n_models, self.n_params)

    # ------------------------------------------------------------------ K0 / K2
    def predict_dev(self, X_dev, out_dev=None, model=0):
        torch = _torch()
        S = X_dev.shape[0]
        assert X_dev.dtype == torch.float32 and X_dev.is_contiguous() and X_dev.shape[1] == self.D
        if out_dev is None:
            out_dev = torch.empty(S, dtype=torch.float32, device=self._tdev())
        _lib.check(self.lib.bore_mlp_predict(self.h, model, _ptr(X_dev), S, _ptr(out_dev),
                                             self._stream()))
        return out_dev

    def predict(self, X, model=0):
        """Keras ``predict`` (bore/mixins.py:50): X (S, D) -> (S, 1) float32."""
        X = np.asarray(X)
        if X.shape[0] == 0:
            return np.zeros((0, 1), np.float32)
        out = self.predict_dev(self.to_device(X, np.float32), model=model)
        return out.cpu().numpy().reshape(-1, 1)

    def value_and_grad_dev(self, X_dev, transform="identity", negate=True, f_dev=None, g_dev=None,
                           model=0):
        torch = _torch()
        S = X_dev.shape[0]
        assert X_dev.dtype == torch.float32 and X_dev.is_contiguous() and X_dev.shape[1] == self.D
        if f_dev is None:
            f_dev = torch.empty(S, dtype=torch.float32, device=self._tdev())
        if g_dev is None:
            g_dev = torch.empty(S, self.D, dtype=torch.float32, device=self._tdev())
        _lib.check(self.lib.bore_mlp_value_and_grad(self.h, model, TRANSFORM_CODES[transform],
                                                    1 if negate else 0, _ptr(X_dev), S,
                                                    _ptr(f_dev), _ptr(g_dev), self._stream()))
        return f_dev, g_dev

    def value_and_grad(self, X, transform="identity", negate=True, model=0):
        """f = T(+-u(x)), g = df/dx for every row of X (float32 results)."""
        X = np.atleast_2d(np.asarray(X))
        f, g = self.value_and_grad_dev(self.to_device(X, np.float32), transform, negate,
                                       model=model)
        return f.cpu().numpy(), g.cpu().numpy()

    # ------------------------------------------------------------------ K3
    def _workspace(self, nbytes):
        torch = _torch()
        if self._work is None or self._work.numel() < nbytes:
            self._work = torch.empty(int(nbytes), dtype=torch.uint8, device=self._tdev())
        return self._work

    def lbfgsb_dev(self, X0_dev, lo, hi, transform="identity", m=10, ftol=1e-9, gtol=1e-5,
                   maxiter=1000, maxfun=15000, maxls=20, model=0):
        """All rows of X0_dev (S, D) float64 minimised on device.  Returns a dict of device
        tensors (x, fun, nit, nfev, status, task) plus ints rounds / evals."""
        torch = _torch()
        S, D = X0_dev.shape
        assert D == self.D and X0_dev.dtype == torch.float64 and X0_dev.is_contiguous()
        lo = np.ascontiguousarray(np.broadcast_to(np.asarray(lo, np.float64), (D,)))
        hi = np.ascontiguousarray(np.broadcast_to(np.asarray(hi, np.float64), (D,)))
        nbytes = self.lib.bore_lbfgsb_minimize_workspace_bytes(self.h, S, m)
        work = self._workspace(nbytes)
        dev = self._tdev()
        x = torch.empty(S, D, dtype=torch.float64, device=dev)
        fun = torch.empty(S, dtype=torch.float64, device=dev)
        ints = torch.empty(4, S, dtype=torch.int32, device=dev)
        rounds, evals = C.c_int(), C.c_longlong()
        _lib.check(self.lib.bore_lbfgsb_minimize(
            self.h, model, TRANSFORM_CODES[transform], _ptr(X0_dev), S, _np_ptr(lo), _np_ptr(hi),
            int(m), float(ftol), float(gtol), int(maxiter), int(maxfun), int(maxls),
            _ptr(work), work.numel(), _ptr(x), _ptr(fun), _ptr(ints[0]), _ptr(ints[1]),
            _ptr(ints[2]), _ptr(ints[3]), C.byref(rounds), C.byref(evals), self._stream()))
        return dict(x=x, fun=fun, nit=ints[0], nfev=ints[1], status=ints[2], task=ints[3],
                    rounds=rounds.value, evals=evals.value)

    def lbfgsb(self, X0, lo, hi, **kw):
        X0 = np.atleast_2d(np.asarray(X0, np.float64))
        r = self.lbfgsb_dev(self.to_device(X0, np.float64), lo, hi, **kw)
        return {k: (v.cpu().numpy() if hasattr(v, "cpu") else v) for k, v in r.items()}

    # ------------------------------------------------------------------ K4
    def topk_smallest(self, f_dev, k, negate=False):
        """Indices (int32, device) of the k smallest entries of f_dev (or of -f_dev), ascending,
        ties by lower index -- np.argpartition's job at bore/mixins.py:56."""
        torch = _torch()
        S = f_dev.shape[0]
        assert f_dev.dtype == torch.float32 and f_dev.is_contiguous()
        idx = torch.empty(int(k), dtype=torch.int32, device=self._tdev())
        nbytes = self.lib.bore_topk_workspace_bytes(S, int(k))
        work = torch.empty(int(nbytes), dtype=torch.uint8, device=self._tdev())
        _lib.check(self.lib.bore_topk_smallest(_ptr(f_dev), S, int(k), 1 if negate else 0, _ptr(idx),
                                               _ptr(work), work.numel(), self.device, self._stream()))
        return idx

    def select_best(self, fun_dev, status_dev, keep_dev=None, idx_offset=0):
        """One int64 (device) packing the first-minimum winner; 0 if no start qualifies."""
        torch = _torch()
        S = fun_dev.shape[0]
        assert fun_dev.dtype == torch.float64 and status_dev.dtype == torch.int32
        key = torch.zeros(1, dtype=torch.int64, device=self._tdev())
        _lib.check(self.lib.bore_select_best(_ptr(fun_dev), _ptr(status_dev), _ptr(keep_dev), S,
                                             int(idx_offset), _ptr(key), self.device, self._stream()))
        return key

    # ------------------------------------------------------------------ batched problems
    def predict_multi_dev(self, X_dev, model0=0):
        """X_dev (M, P, D) float32 -> (M, P) float32, model model0+b on block b."""
        torch = _torch()
        M, P, D = X_dev.shape
        assert D == self.D and X_dev.dtype == torch.float32 and X_dev.is_contiguous()
        out = torch.empty(M, P, dtype=torch.float32, device=self._tdev())
        _lib.check(self.lib.bore_mlp_predict_multi(self.h, int(model0), int(M), _ptr(X_dev), int(P),
                                                   _ptr(out), self._stream()))
        return out

    def topk_groups(self, f_dev, k, negate=False):
        """Per row of f_dev (M, P): indices of the k smallest (of -f when negate), ascending."""
        torch = _torch()
        M, P = f_dev.shape
        assert f_dev.dtype == torch.float32 and f_dev.is_contiguous()
        idx = torch.empty(M, int(k), dtype=torch.int32, device=self._tdev())
        _lib.check(self.lib.bore_topk_smallest_groups(_ptr(f_dev), int(M), int(P), int(k),
                                                      1 if negate else 0, _ptr(idx), self.device,
                                                      self._stream()))
        return idx

    def lbfgsb_multi_dev(self, X0_dev, lo, hi, transform="identity", m=10, ftol=1e-9, gtol=1e-5,
                         maxiter=1000, maxfun=15000, maxls=20, model0=0):
        """X0_dev (M, K, D) float64: K starts for each of M models, all advanced together."""
        torch = _torch()
        M, K, D = X0_dev.shape
        assert D == self.D and X0_dev.dtype == torch.float64 and X0_dev.is_contiguous()
        S = M * K
        lo = np.ascontiguousarray(np.broadcast_to(np.asarray(lo, np.float64), (D,)))
        hi = np.ascontiguousarray(np.broadcast_to(np.asarray(hi, np.float64), (D,)))
        work = self._workspace(self.lib.bore_lbfgsb_minimize_workspace_bytes(self.h, S, m))
        dev = self._tdev()
        x = torch.empty(M, K, D, dtype=torch.float64, device=dev)
        fun = torch.empty(M, K, dtype=torch.float64, device=dev)
        ints = torch.empty(4, M, K, dtype=torch.int32, device=dev)
        rounds, evals = C.c_int(), C.c_longlong()
        _lib.check(self.lib.bore_lbfgsb_minimize_multi(
            self.h, int(model0), int(M), int(K), TRANSFORM_CODES[transform], _ptr(X0_dev),
            _np_ptr(lo), _np_ptr(hi), int(m), float(ftol), float(gtol), int(maxiter), int(maxfun),
            int(maxls), _ptr(work), work.numel(), _ptr(x), _ptr(fun), _ptr(ints[0]), _ptr(ints[1]),
            _ptr(ints[2]), _ptr(ints[3]), C.byref(rounds), C.byref(evals), self._stream()))
        return dict(x=x, fun=fun, nit=ints[0], nfev=ints[1], status=ints[2], task=ints[3],
                    rounds=rounds.value, evals=evals.value)

    def select_best_groups(self, fun_dev, status_dev, keep_dev=None):
        """(M, K) results -> int64 (M,) keys; key & 0x7fffffff = 0x7fffffff - winner's index in
        its group, key 0 = no start of the group qualifies.  ``keep_dev`` (M, K) uint8: filter mask."""
        torch = _torch()
        M, K = fun_dev.shape
        assert fun_dev.dtype == torch.float64 and status_dev.dtype == torch.int32
        assert keep_dev is None or (keep_dev.dtype == torch.uint8 and keep_dev.shape == (M, K))
        keys = torch.empty(M, dtype=torch.int64, device=self._tdev())
        _lib.check(self.lib.bore_select_best_groups(_ptr(fun_dev), _ptr(status_dev), _ptr(keep_dev),
                                                    int(M), int(K), _ptr(keys), self.device,
                                                    self._stream()))
        return keys

    # ------------------------------------------------------------------ data step (section 8f row 2)
    def quantile_labels_dev(self, y_dev, gamma, want_tau=False):
        """y_dev (M, N) float64 -> z (M, N) float32 of 0/1 (and tau (M,)): bore/data.py:31-35 on
        the device for M problems at once."""
        torch = _torch()
        assert y_dev.dtype == torch.float64 and y_dev.dim() == 2 and y_dev.is_contiguous()
        M, N = y_dev.shape
        z = torch.empty(M, N, dtype=torch.float32, device=self._tdev())
        tau = torch.empty(M, dtype=torch.float64, device=self._tdev()) if want_tau else None
        _lib.check(self.lib.bore_quantile_labels(_ptr(y_dev), int(M), int(N), float(gamma), _ptr(z), None,
                                                 _ptr(tau), self.device, self._stream()))
        return (z, tau) if want_tau else z

    def keep_unique_dev(self, x_dev, x_prev_dev, rtol=1e-5, atol=1e-8):
        """x_dev (G, K, D), x_prev_dev (G, N, D) float64 -> keep (G, K) uint8: 0 where the
        candidate is np.allclose to a stored row of its group (bore/data.py:42-48)."""
        torch = _torch()
        G, K, D = x_dev.shape
        assert x_dev.dtype == torch.float64 and x_dev.is_contiguous()
        assert x_prev_dev.dtype == torch.float64 and x_prev_dev.is_contiguous()
        assert x_prev_dev.shape[0] == G and x_prev_dev.shape[2] == D
        keep = torch.empty(G, K, dtype=torch.uint8, device=self._tdev())
        _lib.check(self.lib.bore_is_duplicate(_ptr(x_dev), int(G), int(K), _ptr(x_prev_dev),
                                              int(x_prev_dev.shape[1]), int(D), float(rtol), float(atol),
                                              None, _ptr(keep), self.device, self._stream()))
        return keep

    def quantile_labels_ragged_dev(self, y_dev, n, gamma, want_tau=False):
        """y_dev (sum n_p,) float64, the targets of M problems one after the other, n (M,) their
        counts -> z (sum n_p,) float32 of 0/1 (and tau (M,)): every problem labelled over its own
        targets (bore_quantile_labels_ragged)."""
        torch = _torch()
        n = np.ascontiguousarray(n, np.int32)
        assert y_dev.dtype == torch.float64 and y_dev.dim() == 1 and y_dev.is_contiguous()
        assert y_dev.shape[0] == int(n.astype(np.int64).sum())
        z = torch.empty(y_dev.shape[0], dtype=torch.float32, device=self._tdev())
        tau = torch.empty(len(n), dtype=torch.float64, device=self._tdev()) if want_tau else None
        _lib.check(self.lib.bore_quantile_labels_ragged(_ptr(y_dev), len(n), _np_ptr(n), float(gamma), _ptr(z),
                                                        None, _ptr(tau), self.device, self._stream()))
        return (z, tau) if want_tau else z

    def keep_unique_ragged_dev(self, x_dev, n_prev, x_prev_dev, rtol=1e-5, atol=1e-8):
        """x_dev (G, K, D) float64, n_prev (G,) stored rows per group (0 allowed), x_prev_dev
        (sum n_prev, D) float64 the groups' rows one group after the other -> keep (G, K) uint8
        (bore_is_duplicate_ragged)."""
        torch = _torch()
        G, K, D = x_dev.shape
        n_prev = np.ascontiguousarray(n_prev, np.int32)
        assert x_dev.dtype == torch.float64 and x_dev.is_contiguous() and len(n_prev) == G
        assert x_prev_dev.dtype == torch.float64 and x_prev_dev.is_contiguous()
        assert tuple(x_prev_dev.shape) == (int(n_prev.astype(np.int64).sum()), D)
        keep = torch.empty(G, K, dtype=torch.uint8, device=self._tdev())
        _lib.check(self.lib.bore_is_duplicate_ragged(_ptr(x_dev), int(G), int(K),
                                                     _ptr(x_prev_dev) if x_prev_dev.numel() else None,
                                                     _np_ptr(n_prev), int(D), float(rtol), float(atol), None,
                                                     _ptr(keep), self.device, self._stream()))
        return keep

    def distort_dev(self, loc_dev, distortion, low, high, u_dev):
        """loc_dev (P, D) float64 suggestions -> truncated-normal resamples around them
        (bore/base.py:45-64) from the uniform variates u_dev (P, D) drawn on the host."""
        torch = _torch()
        P, D = loc_dev.shape
        assert loc_dev.dtype == torch.float64 and loc_dev.is_contiguous()
        assert u_dev.shape == (P, D) and u_dev.dtype == torch.float64 and u_dev.is_contiguous()
        lo = self.to_device(np.broadcast_to(np.asarray(low, np.float64), (D,)), np.float64)
        hi = self.to_device(np.broadcast_to(np.asarray(high, np.float64), (D,)), np.float64)
        out = torch.empty_like(loc_dev)
        _lib.check(self.lib.bore_truncnorm_distort(_ptr(loc_dev), int(P), int(D), float(distortion), _ptr(lo),
                                                   _ptr(hi), _ptr(u_dev), _ptr(out), self.device, self._stream()))
        return out

    # ------------------------------------------------------------------ SVGD (section 8f row 3)
    def svgd_maximize(self, x_init, transform, low, high, n_iter, length_scale, step_size, alpha, eps,
                      tau, lambd, zeta_c, model0=0):
        """x_init (n, D) or (P, n, D) float64 -> particles after n_iter SVGD iterations on
        transform(model(x)) (maximised), model model0+p for block p; the whole loop is enqueued
        at once (bore_svgd_maximize)."""
        torch = _torch()
        x = np.asarray(x_init, np.float64)
        single = x.ndim == 2
        x3 = x[None] if single else x
        P, n, D = x3.shape
        assert D == self.D and model0 + P <= self.n_models
        x_dev = self.to_device(x3, np.float64).clone()
        nbytes = self.lib.bore_svgd_workspace_bytes(P, n, D)
        work = torch.empty(int(nbytes), dtype=torch.uint8, device=self._tdev())
        lo = hi = None
        if low is not None:
            lo = np.ascontiguousarray(np.broadcast_to(np.asarray(low, np.float64), (D,)))
            hi = np.ascontiguousarray(np.broadcast_to(np.asarray(high, np.float64), (D,)))
        _lib.check(self.lib.bore_svgd_maximize(
            self.h, int(model0), int(P), TRANSFORM_CODES[transform], _ptr(x_dev), int(n),
            _np_ptr(lo) if lo is not None else None, _np_ptr(hi) if hi is not None else None,
            float(length_scale), int(n_iter), float(step_size), float(alpha), float(eps), float(tau),
            float(lambd), float(zeta_c), _ptr(work), work.numel(), self._stream()))
        out = x_dev.cpu().numpy()
        return out[0] if single else out

    # ------------------------------------------------------------------ K1
    def fit_dev(self, X_dev, z_dev, N, batch_size, epochs, perm_dev, loss_dev=None,
                model0=0, count=1, shared_data=True, shared_perm=True, w_dev=None, class_weight=None):
        """``w_dev`` (float32, the layout of ``z_dev``) and ``class_weight`` ((weight of label 0,
        weight of label 1)) weight each sample's loss (bore_mlp_fit_weighted); without them this
        is bore_mlp_fit."""
        torch = _torch()
        assert X_dev.dtype == torch.float32 and z_dev.dtype == torch.float32
        assert perm_dev.dtype == torch.int32 and perm_dev.is_contiguous()
        if loss_dev is None:
            loss_dev = torch.empty(count, epochs, dtype=torch.float32, device=self._tdev())
        if w_dev is None and class_weight is None:
            _lib.check(self.lib.bore_mlp_fit(self.h, model0, count, _ptr(X_dev), _ptr(z_dev), int(N),
                                             1 if shared_data else 0, int(batch_size), int(epochs),
                                             _ptr(perm_dev), 1 if shared_perm else 0,
                                             _ptr(loss_dev), self._stream()))
            return loss_dev
        assert w_dev is None or (w_dev.dtype == torch.float32 and w_dev.is_contiguous()
                                 and w_dev.numel() == z_dev.numel())
        cw0, cw1 = (1.0, 1.0) if class_weight is None else class_weight
        _lib.check(self.lib.bore_mlp_fit_weighted(self.h, model0, count, _ptr(X_dev), _ptr(z_dev), _ptr(w_dev),
                                                  int(N), 1 if shared_data else 0, float(cw0), float(cw1),
                                                  int(batch_size), int(epochs), _ptr(perm_dev),
                                                  1 if shared_perm else 0, _ptr(loss_dev), self._stream()))
        return loss_dev

    def fit_ragged_dev(self, X_dev, z_dev, layout, batch_size, perm_dev, model0=0, w_dev=None,
                       class_weight=None):
        """Problems model0 .. model0 + M - 1 with their own observation counts and epochs
        (``layout``: a ``ragged.RaggedLayout``) in one launch (bore_mlp_fit_ragged).  X_dev
        (sum N_p, D), z_dev / w_dev (sum N_p,) float32 and perm_dev (sum epochs_p * N_p,) int32 hold
        the problems one after the other.  Returns the concatenated epoch losses (sum epochs_p,)."""
        torch = _torch()
        assert X_dev.dtype == torch.float32 and z_dev.dtype == torch.float32
        assert perm_dev.dtype == torch.int32 and perm_dev.is_contiguous()
        n = np.ascontiguousarray(layout.n, np.int32)
        e = np.ascontiguousarray(layout.epochs, np.int32)
        R, Q, E = int(layout.rows[-1]), int(layout.perms[-1]), int(layout.losses[-1])
        assert X_dev.shape == (R, self.D) and z_dev.numel() == R and perm_dev.numel() == Q
        assert w_dev is None or (w_dev.dtype == torch.float32 and w_dev.is_contiguous() and w_dev.numel() == R)
        if Q == 0:  # nothing trains; the call still checks its arguments
            perm_dev = torch.zeros(1, dtype=torch.int32, device=self._tdev())
        loss_dev = torch.empty(max(E, 1), dtype=torch.float32, device=self._tdev())
        cw0, cw1 = (1.0, 1.0) if class_weight is None else class_weight
        _lib.check(self.lib.bore_mlp_fit_ragged(self.h, int(model0), len(n), _ptr(X_dev), _ptr(z_dev), _ptr(w_dev),
                                                _np_ptr(n), _np_ptr(e), float(cw0), float(cw1), int(batch_size),
                                                _ptr(perm_dev), _ptr(loss_dev), self._stream()))
        return loss_dev[:E]

    def fit(self, X, z, epochs, batch_size, permutations, l2=None, model=0, w=None, class_weight=None):
        """Keras ``fit`` with explicit per-epoch permutations -> history loss (epochs,).
        ``w`` (N,) sample weights and ``class_weight`` (cw0, cw1) as in ``fit_dev``."""
        if l2 is not None:
            self.set_regularizers(l2)
        X = np.asarray(X)
        N = X.shape[0]
        perm = np.ascontiguousarray(permutations, np.int32).reshape(epochs, N)
        return self.fit_async(X, z, epochs, batch_size, perm, model=model, w=w,
                              class_weight=class_weight).cpu().numpy()[0]

    def fit_async(self, X, z, epochs, batch_size, permutations, l2=None, model=0, w=None, class_weight=None):
        """Like ``fit`` but returns the (1, epochs) device tensor of epoch losses without waiting
        for the training kernel: the host is free (e.g. to draw the start points of the next
        argmax) while the GPU trains."""
        if l2 is not None:
            self.set_regularizers(l2)
        X = np.asarray(X)
        N = X.shape[0]
        perm = np.ascontiguousarray(permutations, np.int32).reshape(epochs, N)
        w_dev = None if w is None else self.to_device(np.asarray(w, np.float32).reshape(N), np.float32)
        return self.fit_dev(self.to_device(X, np.float32),
                            self.to_device(np.asarray(z).astype(np.float32), np.float32),
                            N, batch_size, epochs, self.to_device(perm, np.int32),
                            model0=model, count=1, w_dev=w_dev, class_weight=class_weight)

    def evaluate(self, X, z, l2=None, model=0, w=None, class_weight=None):
        """Keras ``evaluate`` -> [loss, accuracy]; ``w`` / ``class_weight`` weight the loss and the
        accuracy (bore_mlp_evaluate_weighted)."""
        if l2 is not None:
            self.set_regularizers(l2)
        X = np.asarray(X)
        N = X.shape[0]
        out = np.zeros(2, np.float32)
        Xd = self.to_device(X, np.float32)
        zd = self.to_device(np.asarray(z).astype(np.float32), np.float32)
        if w is None and class_weight is None:
            _lib.check(self.lib.bore_mlp_evaluate(self.h, model, _ptr(Xd), _ptr(zd), N,
                                                  _np_ptr(out), self._stream()))
        else:
            wd = None if w is None else self.to_device(np.asarray(w, np.float32).reshape(N), np.float32)
            cw0, cw1 = (1.0, 1.0) if class_weight is None else class_weight
            _lib.check(self.lib.bore_mlp_evaluate_weighted(self.h, model, _ptr(Xd), _ptr(zd), _ptr(wd),
                                                           float(cw0), float(cw1), N, _np_ptr(out),
                                                           self._stream()))
        return [float(out[0]), float(out[1])]


def ffma_peak_tflops(device=0, iters=4096):
    lib = _lib.require_cuda()
    out = C.c_double()
    _lib.check(lib.bore_bench_ffma_peak(int(device), int(iters), C.byref(out)))
    return out.value


# ---------------------------------------------------------------------- SVGD without a model handle
def _current_device():
    lib = _lib.require_cuda()
    torch = _torch()
    if not torch.cuda.is_available():
        raise _lib.BoreNativeError("torch sees no CUDA device; bore_b200 has no CPU fallback")
    dev = torch.cuda.current_device()
    return lib, torch, dev, torch.device("cuda", dev), C.c_void_p(torch.cuda.current_stream(dev).cuda_stream)


def svgd_kernel_value_and_grad(X, length_scale):
    """RadialBasis.value_and_grad on the device: X (n, D) float64 -> K (n, n), K_grad (n, D)."""
    lib, torch, dev, tdev, stream = _current_device()
    X = np.ascontiguousarray(X, np.float64)
    n, D = X.shape
    x_dev = torch.from_numpy(X).to(tdev)
    K = torch.empty(n, n, dtype=torch.float64, device=tdev)
    Kg = torch.empty(n, D, dtype=torch.float64, device=tdev)
    ls = float("nan") if length_scale is None else float(length_scale)
    _lib.check(lib.bore_svgd_kernel_value_and_grad(_ptr(x_dev), n, D, ls, _ptr(K), _ptr(Kg), dev, stream))
    return K.cpu().numpy(), Kg.cpu().numpy()


class SvgdStepper:
    """Device-resident SVGD state (particles + AdaGrad accumulator) advanced one iteration at a
    time with a caller-supplied ``f, f_grad`` (bore_svgd_step) -- for objectives that are not a
    bore_b200 model (the reference's SVGD accepts any callable, svgd/base.py:78)."""

    def __init__(self, x_init, low, high, length_scale, step_size, alpha, eps, tau, lambd, zeta_c):
        self.lib, torch, self.dev, tdev, _ = _current_device()
        x = np.ascontiguousarray(x_init, np.float64)
        assert x.ndim == 2
        self.n, self.D = x.shape
        self._x = torch.from_numpy(x).to(tdev)
        self._hist = torch.zeros_like(self._x)
        self._lo = self._hi = None
        if low is not None:
            D = self.D
            self._lo = torch.from_numpy(np.array(np.broadcast_to(np.asarray(low, np.float64), (D,)))).to(tdev)
            self._hi = torch.from_numpy(np.array(np.broadcast_to(np.asarray(high, np.float64), (D,)))).to(tdev)
        self._opts = (float(length_scale), float(step_size), float(alpha), float(eps), float(tau),
                      float(lambd), float(zeta_c))
        self._it = 0
        self._tdev = tdev

    def x(self):
        return self._x.cpu().numpy()

    def step(self, f, f_grad):
        torch = _torch()
        f = np.array(np.broadcast_to(f, (self.n,)), np.float64)
        g = np.array(f_grad, np.float64)
        assert g.shape == (self.n, self.D)
        f_dev, g_dev = torch.from_numpy(f).to(self._tdev), torch.from_numpy(g).to(self._tdev)
        ls, step, alpha, eps, tau, lambd, zc = self._opts
        stream = C.c_void_p(torch.cuda.current_stream(self.dev).cuda_stream)
        _lib.check(self.lib.bore_svgd_step(_ptr(self._x), 1, self.n, self.D, _ptr(f_dev), _ptr(g_dev), 1,
                                           _ptr(self._lo), _ptr(self._hi), ls, self._it, step, alpha, eps,
                                           tau, lambd, zc, _ptr(self._hist), None, self.dev, stream))
        self._it += 1
