"""Shared synthetic problems for the parity tests (seeded, oracle-sized)."""
import numpy as np

from oracle import keras_mlp as km

# (name, dims, activations, transform) -- the BASELINE.json configs' networks
NETS = {
    "cfg1_branin": ([2, 16, 16, 1], ["relu", "relu", "sigmoid"], "identity"),
    "cfg2_hartmann6": ([6, 32, 32, 1], ["relu", "relu", "sigmoid"], "identity"),
    "cfg3_ackley50": ([50, 64, 64, 64, 1], ["relu", "relu", "relu", "sigmoid"], "identity"),
    "cfg5_plugin8": ([8, 32, 32, 32, 1], ["elu", "elu", "elu", "linear"], "sigmoid"),
    "ref_test_linear": ([2, 32, 32, 32, 1], ["linear"] * 4, "identity"),
    "tanh_exp": ([5, 24, 40, 1], ["tanh", "sigmoid", "linear"], "exp"),
    "no_hidden": ([7, 1], ["sigmoid"], "identity"),
}


def synthetic_targets(X):
    """Smooth multimodal test objective on the unit cube (stand-in for Branin/Hartmann/Ackley)."""
    return np.sum((X - 0.4) ** 2, axis=1) + 0.1 * np.sin(5.0 * X[:, 0]) * np.cos(3.0 * X[:, -1])


def lstm_sequences(seed, N, T, D, mask_value):
    """Padded per-rung sequences X (N, T, D), Y (N, T, 1) as the multi-fidelity record makes them: every
    sequence stops at a random rung, every third may start one rung late, some have a masked gap."""
    rs = np.random.RandomState(seed)
    X = rs.uniform(size=(N, T, D))
    Y = (rs.uniform(size=(N, T, 1)) < 0.4).astype(np.float64)
    for n in range(N):
        first = rs.randint(0, 2) if n % 3 == 0 and T > 1 else 0      # brackets that start at a higher budget
        keep = rs.randint(first + 1, T + 1)
        X[n, :first] = mask_value; Y[n, :first] = mask_value
        X[n, keep:] = mask_value; Y[n, keep:] = mask_value
        if n % 7 == 3 and keep - first > 2:
            X[n, first + 1] = mask_value; Y[n, first + 1] = mask_value   # a gap
    return X, Y


def lstm_factory(D, U, L, activation, seed=0, l2f=None):
    """StackedRecurrentFactory of L cells of U units on D inputs, l2(l2f) on the kernels and biases."""
    from bore_b200.layers import l2
    from bore_b200.models import StackedRecurrentFactory
    reg = None if l2f is None else l2(l2f)
    return StackedRecurrentFactory(D, 1, num_layers=L, num_units=U, seed=seed,
                                   layer_kws=dict(activation=activation, kernel_regularizer=reg,
                                                  bias_regularizer=reg))


def trained_weights(dims, acts, seed=0, N=300, epochs=30, gamma=0.25):
    """Glorot init + a short oracle fit on quantile-labelled data: realistic, non-degenerate
    weights for value/gradient/argmax parity."""
    rs = np.random.RandomState(seed)
    w = km.init_weights(dims, seed)
    X = rs.uniform(size=(N, dims[0]))
    y = synthetic_targets(X)
    z = y < np.quantile(y, gamma)
    perms = np.array([rs.permutation(N) for _ in range(epochs)])
    acts_fit = list(acts)
    if acts_fit[-1] not in ("sigmoid", "linear"):
        acts_fit[-1] = "linear"
    km.fit(w, acts_fit, X, z, epochs, 64, perms)
    return w


def permuted_units(weights, seed=0):
    """The same network with the hidden units of every hidden layer permuted: mathematically the
    identical function, but every dot product is summed in a different order -- an fp32
    re-association of the kind any other implementation of the same MLP (TensorFlow's Eigen
    kernels, this NumPy oracle, a CUDA kernel) differs by."""
    rs = np.random.RandomState(seed)
    ws = [np.array(w) for w in weights]
    n_layers = len(ws) // 2
    for l in range(n_layers - 1):
        perm = rs.permutation(ws[2 * l].shape[1])
        ws[2 * l] = ws[2 * l][:, perm]
        ws[2 * l + 1] = ws[2 * l + 1][perm]
        ws[2 * l + 2] = ws[2 * l + 2][perm, :]
    return ws


def reference_self_agreement(weights, acts, X0, bounds, transform, tol, ref=None):
    """Fraction of starts on which the reference path (oracle MLP + SciPy L-BFGS-B) reaches the
    same objective value (within tol) as ITSELF after an fp32 re-association of the MLP.  On
    piecewise-linear (ReLU) objectives this is well below 1 -- the yardstick for what "agrees
    with the reference" can mean there (SURVEY.md 7.2.1)."""
    from oracle import argmax as am
    if ref is None:
        ref = am.minimize_starts(weights, acts, X0, bounds, transform=transform)
    alt = am.minimize_starts(permuted_units(weights), acts, X0, bounds, transform=transform)
    return float(np.mean(np.abs(alt["fun"] - ref["fun"]) <= tol)), ref, alt


class fork_pool:
    """``multiprocessing`` pool of FORKED workers (NumPy / SciPy only) next to a parent that has CUDA
    initialised.  A forked child must never run a destructor that touches CUDA (torch tensors, events,
    native handles): if the child's garbage collector finds such objects in an unreachable cycle -- models hold
    one through their ``convert`` closure -- the CUDA runtime aborts the child and the pool hangs.  So the
    parent collects its garbage first and FREEZES what is alive (``gc.freeze``: the child's collector never
    looks at it); the handles additionally ignore ``__del__`` in a process that did not create them."""

    def __init__(self, cores):
        import gc
        import multiprocessing as mp
        gc.collect()
        gc.freeze()
        try:
            self.pool = mp.get_context("fork").Pool(cores)
        finally:
            gc.unfreeze()

    def __enter__(self):
        return self.pool

    def __exit__(self, *exc):
        self.pool.terminate()
        self.pool.join()
        return False


def _minimize_chunk(args):
    weights, acts, X0, lo, hi, transform, options = args
    from scipy.optimize import Bounds
    from threadpoolctl import threadpool_limits
    from oracle import argmax as am
    with threadpool_limits(1):  # batch-of-1 matmuls: BLAS threads only add contention
        return am.minimize_starts(weights, acts, X0, Bounds(lo, hi), options=options, transform=transform)


def parallel_minimize_starts(weights, acts, X0, lo, hi, transform, options=dict(maxiter=1000, ftol=1e-9)):
    """oracle.argmax.minimize_starts with the starts spread over the host cores (one
    scipy.optimize.minimize per start, as the reference runs them; starts are independent)."""
    import multiprocessing as mp
    import os
    cores = max(1, min(os.cpu_count() or 1, 32))
    n = X0.shape[1]
    lo = np.broadcast_to(np.asarray(lo, np.float64), (n,)).copy()
    hi = np.broadcast_to(np.asarray(hi, np.float64), (n,)).copy()
    jobs = [(weights, acts, c, lo, hi, transform, options) for c in np.array_split(X0, 2 * cores) if len(c)]
    if cores == 1:
        outs = [_minimize_chunk(j) for j in jobs]
    else:
        with fork_pool(cores) as pool:
            outs = pool.map(_minimize_chunk, jobs)
    return {k: np.concatenate([o[k] for o in outs]) for k in outs[0]}
