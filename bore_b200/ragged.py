"""Host-side layout of ragged batched problems: M problems that each hold their own number of
observations N_p and train for their own number of epochs (``BatchedMaximizableSequential.fit`` with
lists, ``bore_mlp_fit_ragged``).  Pure NumPy: every shape check happens here, before anything reaches
the device.

The problems' arrays are concatenated in problem order.  With the 64-bit prefix sums
    rows[p]  = sum_{q<p} N_q             first row of problem p in X / y / sample weights
    perms[p] = sum_{q<p} epochs_q * N_q  first entry of its (epochs_p, N_p) permutations
    losses[p] = sum_{q<p} epochs_q       first of its epoch losses
problem p's data are X[rows[p]:rows[p+1]] and so on; the device kernels read the same offsets.
"""
import numpy as np


class RaggedLayout:
    """Counts and offsets of M ragged problems.  ``n`` (M,) observation counts >= 1, ``epochs`` (M,)
    epoch counts >= 0; ``rows``, ``perms``, ``losses``: the (M + 1,) int64 prefix sums above."""

    def __init__(self, n, epochs):
        self.n = np.asarray(n, np.int64).reshape(-1)
        self.epochs = np.asarray(epochs, np.int64).reshape(-1)
        if self.n.shape != self.epochs.shape or len(self.n) == 0:
            raise ValueError(f"{len(self.n)} observation counts and {len(self.epochs)} epoch counts")
        if (self.n < 1).any():
            raise ValueError(f"every problem needs at least one observation, got N = {self.n.min()}")
        if (self.epochs < 0).any():
            raise ValueError(f"epochs must be >= 0, got {self.epochs.min()}")
        if self.n.max() > np.iinfo(np.int32).max or self.epochs.max() > np.iinfo(np.int32).max:
            raise ValueError("observation and epoch counts must fit 32 bits")
        zero = np.zeros(1, np.int64)
        self.rows = np.concatenate([zero, np.cumsum(self.n)])
        self.perms = np.concatenate([zero, np.cumsum(self.n * self.epochs)])
        self.losses = np.concatenate([zero, np.cumsum(self.epochs)])

    def __len__(self):
        return len(self.n)

    def steps(self, batch_size):
        """Adam steps of every problem: epochs_p * ceil(N_p / batch_size)."""
        return self.epochs * (-(-self.n // int(batch_size)))

    def pad_loss(self, flat):
        """The concatenated epoch losses (sum of epochs_p,) -> (M, max epochs_p), NaN beyond each
        problem's epochs."""
        flat = np.asarray(flat)
        assert flat.shape == (int(self.losses[-1]),)
        out = np.full((len(self), int(self.epochs.max())), np.nan, flat.dtype if flat.size else np.float32)
        for p in range(len(self)):
            out[p, :self.epochs[p]] = flat[self.losses[p]:self.losses[p + 1]]
        return out


def _as_list(name, v, M):
    if not isinstance(v, (list, tuple)) or len(v) != M:
        got = f"{len(v)} entries" if isinstance(v, (list, tuple)) else type(v).__name__
        raise ValueError(f"{name} must be a list of {M} arrays, one per problem; got {got}")
    return v


def ragged_inputs(x, y, n_problems, dim, epochs, sample_weight=None, permutations=None,
                  random_state=None, shuffle=True):
    """Checks and concatenates the list form of a batched ``fit``.

    ``x``: M arrays (N_p, dim); ``y``: M arrays (N_p,); ``epochs``: an int or M ints;
    ``sample_weight``: None or M arrays (N_p,) (or (N_p, 1)); ``permutations``: None or M arrays
    (epochs_p, N_p).  Without permutations they are drawn from ``random_state`` problem after problem,
    epoch after epoch, ``permutation(N_p)`` -- the order of the uniform call -- or are the identity
    when ``shuffle`` is false.  Raises ValueError on every shape or length error.

    Returns ``(layout, X (sum N_p, dim), y (sum N_p,), w (sum N_p,) float32 or None,
    perm (sum epochs_p * N_p,) int32)``."""
    M = int(n_problems)
    xs = _as_list("x", x, M)
    ys = _as_list("y", y, M)
    xs = [np.asarray(a) for a in xs]
    ys = [np.asarray(a) for a in ys]
    for p, (a, b) in enumerate(zip(xs, ys)):
        if a.ndim != 2 or a.shape[1] != dim or a.shape[0] < 1:
            raise ValueError(f"x[{p}] must have shape (N_p >= 1, {dim}), got {a.shape}")
        if b.shape != (a.shape[0],):
            raise ValueError(f"y[{p}] must have shape ({a.shape[0]},), got {b.shape}")
    n = [a.shape[0] for a in xs]
    ep = [epochs] * M if np.ndim(epochs) == 0 else list(epochs)
    if len(ep) != M:
        raise ValueError(f"epochs must be an int or {M} ints, got {len(ep)}")
    if any(int(e) != e for e in ep):
        raise ValueError(f"epochs must be integers, got {epochs}")
    ep = [int(e) for e in ep]
    layout = RaggedLayout(n, ep)
    w = None
    if sample_weight is not None:
        sws = _as_list("sample_weight", sample_weight, M)
        parts = []
        for p, s in enumerate(sws):
            s = np.asarray(s, np.float32)
            if s.shape not in ((n[p],), (n[p], 1)):
                raise ValueError(f"sample_weight[{p}] must have shape ({n[p]},), got {s.shape}")
            parts.append(s.reshape(n[p]))
        w = np.concatenate(parts)
    if permutations is None:
        if shuffle:
            if random_state is None:
                raise ValueError("shuffling needs a random_state")
            perm = [random_state.permutation(n[p]) for p in range(M) for _ in range(ep[p])]
        else:
            perm = [np.arange(n[p]) for p in range(M) for _ in range(ep[p])]
    else:
        perm = []
        for p, a in enumerate(_as_list("permutations", permutations, M)):
            a = np.asarray(a)
            if a.shape != (ep[p], n[p]):
                raise ValueError(f"permutations[{p}] must have shape ({ep[p]}, {n[p]}), got {a.shape}")
            if a.size and (a.min() < 0 or a.max() >= n[p]):
                raise ValueError(f"permutations[{p}] holds indices outside [0, {n[p]})")
            perm.append(a.reshape(-1))
    perm = np.concatenate(perm).astype(np.int32) if perm else np.zeros(0, np.int32)
    return layout, np.concatenate(xs), np.concatenate(ys), w, perm


def ragged_rows(arrays, n_groups, dim, name="exclude"):
    """M arrays (n_p, dim) with n_p >= 0 -> (counts (M,) int64, rows (sum n_p, dim) float64)."""
    arrs = _as_list(name, arrays, int(n_groups))
    out = []
    for p, a in enumerate(arrs):
        a = np.asarray(a, np.float64)
        if a.size == 0:
            a = a.reshape(0, dim)
        if a.ndim != 2 or a.shape[1] != dim:
            raise ValueError(f"{name}[{p}] must have shape (n_p, {dim}), got {a.shape}")
        out.append(a)
    counts = np.array([a.shape[0] for a in out], np.int64)
    return counts, np.concatenate(out)
