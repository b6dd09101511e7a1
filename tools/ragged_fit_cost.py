"""What ragged batched training costs, and that it costs the uniform fit nothing.

Times fits with CUDA events, best of --reps after one warm-up launch each:
  cfg3         one [50, 64, 64, 64, 1] ReLU model, N = 2,000, 31 epochs x 32 steps = 992 Adam steps, fit mode 4
  cfg4         4,096 [6, 32, 32, 1] ReLU models, each on its own N = 500, 125 epochs x 8 steps, fit mode 1
  ragged_cfg4  the cfg-4 net on 4,096 Hartmann-6 problems with N_p uniform in [250, 750] and the plugin's rule
               epochs_p = 1000 // ceil(N_p / 64) (bore_mlp_fit_ragged, mode 1)
  skewed       4,096 problems with N_p log-uniform in [10, 2,000], 10 epochs each, launched longest first and
               in problem order (BORE_FIT_RAGGED_ORDER=0)
cfg3 and cfg4 go through bore_mlp_fit, and a digest of the trained weights and Adam state after the warm-up
launch is printed with them: two builds that compute the same bits print the same digests.  The ragged
workloads run when the library has bore_mlp_fit_ragged.  Prints one JSON line with the device name and power
limit.

--lib PATH times another build of libbore_b200.so (e.g. the parent commit's) through the same Python code, so
that two builds can be compared in one session, alternating processes:
  for i in 1 2 3; do python tools/ragged_fit_cost.py --lib OLD.so; python tools/ragged_fit_cost.py; done
"""
import argparse
import hashlib
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.dirname(ROOT))
import numpy as np  # noqa: E402

from weighted_fit_cost import glorot, use_library  # noqa: E402

CFG4_NET = ([6, 32, 32, 1], ["relu", "relu", "sigmoid"])


def hartmann6(X):
    A = np.array([[10, 3, 17, 3.5, 1.7, 8], [0.05, 10, 17, 0.1, 8, 14], [3, 3.5, 1.7, 10, 17, 8],
                  [17, 8, 0.05, 10, 0.1, 14]])
    P = 1e-4 * np.array([[1312, 1696, 5569, 124, 8283, 5886], [2329, 4135, 8307, 3736, 1004, 9991],
                         [2348, 1451, 3522, 2883, 3047, 6650], [4047, 8828, 8732, 5743, 1091, 381]])
    alpha = np.array([1.0, 1.2, 3.0, 3.2])
    return -np.sum(alpha * np.exp(-np.sum(A * (X[:, None, :] - P) ** 2, axis=2)), axis=1)


def _timed(net, launch, reps):
    """Best of `reps` timed launches after one warm-up, each from a zeroed optimizer; digest of the state
    after the warm-up launch."""
    import torch
    times, digest = [], None
    for r in range(reps + 1):
        net.reset_optimizer()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        launch()
        e1.record()
        torch.cuda.synchronize()
        if r:
            times.append(e0.elapsed_time(e1))
        else:
            h = hashlib.sha256(net.params_tensor().cpu().numpy().tobytes())
            m, v, t = net.get_adam_state(model=0)
            h.update(b"".join(a.tobytes() for a in m + v) + str(t).encode())
            digest = h.hexdigest()[:16]
    return min(times), digest


def time_uniform(dims, acts, M, N, E, mode, reps):
    from bore_b200.engine import NativeMLP
    rs = np.random.RandomState(0)
    X = rs.uniform(size=(M * N, dims[0])).astype(np.float32)
    y = np.sum((X - 0.4) ** 2, axis=1).reshape(M, N)
    z = (y < np.quantile(y, 0.25, axis=1, keepdims=True)).astype(np.float32).reshape(-1)
    perm = np.stack([rs.permutation(N) for _ in range(E)]).astype(np.int32)
    net = NativeMLP(dims, acts, n_models=M)
    net.set_fit_mode(mode)
    w0 = glorot(dims, rs)
    for i in range(M):
        net.set_weights(w0, model=i)
    Xd, zd, pd = net.to_device(X, np.float32), net.to_device(z, np.float32), net.to_device(perm, np.int32)
    return _timed(net, lambda: net.fit_dev(Xd, zd, N, 64, E, pd, model0=0, count=M, shared_data=M == 1,
                                           shared_perm=True), reps)


def ragged_case(n, epochs, seed):
    """Device inputs of a ragged cfg-4 launch: Hartmann-6 problems with N_p = n[p] observations."""
    from bore_b200.engine import NativeMLP
    from bore_b200.ragged import RaggedLayout
    dims, acts = CFG4_NET
    rs = np.random.RandomState(seed)
    lay = RaggedLayout(n, epochs)
    X = rs.uniform(size=(int(lay.rows[-1]), 6))
    y = hartmann6(X)
    z = np.concatenate([y[a:b] < np.quantile(y[a:b], 1 / 3) for a, b in zip(lay.rows[:-1], lay.rows[1:])])
    perm = np.concatenate([rs.permutation(int(n[p])) for p in range(len(n)) for _ in range(int(epochs[p]))])
    net = NativeMLP(dims, acts, n_models=len(n))
    net.set_fit_mode(1)
    w0 = glorot(dims, rs)
    for i in range(len(n)):
        net.set_weights(w0, model=i)
    args = (net.to_device(X, np.float32), net.to_device(z.astype(np.float32), np.float32), lay, 64,
            net.to_device(perm.astype(np.int32), np.int32))
    return net, args


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--lib", help="another build of libbore_b200.so to time")
    ap.add_argument("--reps", type=int, default=5)
    args = ap.parse_args()
    if args.lib:
        use_library(args.lib)
    from bore_b200 import _lib
    _lib.require_cuda()
    out = {"lib": args.lib or "tree"}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30)
        out["gpu"] = q.stdout.strip().splitlines()[0]
    except (OSError, subprocess.SubprocessError, IndexError):
        out["gpu"] = "unknown"
    cfg3 = ([50, 64, 64, 64, 1], ["relu", "relu", "relu", "sigmoid"], 1, 2000, 31, 4)
    cfg4 = CFG4_NET + (4096, 500, 125, 1)
    for name, cfg in (("cfg3_mode4", cfg3), ("cfg4_mode1", cfg4)):
        ms, digest = time_uniform(*cfg, args.reps)
        out[name + "_ms"], out[name + "_digest"] = round(ms, 3), digest
    if "bore_mlp_fit_ragged" in _lib.SIGNATURES:
        rs = np.random.RandomState(1)
        n = rs.randint(250, 751, size=4096)
        e = 1000 // -(-n // 64)
        net, a = ragged_case(n, e, seed=2)
        out["ragged_cfg4_ms"] = round(_timed(net, lambda: net.fit_ragged_dev(*a), args.reps)[0], 3)
        out["ragged_cfg4_adam_steps"] = int((e * -(-n // 64)).sum())
        n = np.exp(rs.uniform(np.log(10), np.log(2000), size=4096)).astype(np.int64)
        e = np.full(4096, 10)
        net, a = ragged_case(n, e, seed=3)
        for order in ("1", "0", "1", "0"):  # alternating: longest first, problem order
            os.environ["BORE_FIT_RAGGED_ORDER"] = order
            ms = round(_timed(net, lambda: net.fit_ragged_dev(*a), args.reps)[0], 3)
            key = "skewed_longest_first_ms" if order == "1" else "skewed_problem_order_ms"
            out[key] = min(out.get(key, ms), ms)
        os.environ.pop("BORE_FIT_RAGGED_ORDER")
        out["skewed_adam_steps"] = int((e * -(-n // 64)).sum())
    print(json.dumps(out), flush=True)


if __name__ == "__main__":
    main()
