"""What weighted training costs, and that it costs the unweighted fit nothing.

Times two fits with CUDA events, best of --reps after one warm-up launch each:
  cfg3  one [50, 64, 64, 64, 1] ReLU model, N = 2,000, 31 epochs x 32 steps = 992 Adam steps, fit mode 4 (K1u)
  cfg4  4,096 [6, 32, 32, 1] ReLU models, each on its own N = 500, 125 epochs x 8 steps, fit mode 1 (one CTA each)
unweighted (bore_mlp_fit) and, when the library has it, weighted (bore_mlp_fit_weighted: per-sample weights in
[0, 2) and class weights (0.5, 2.0)).  Prints one JSON line with the device name and power limit.

--lib PATH times another build of libbore_b200.so (e.g. the parent commit's) through the same Python code, so
that two builds can be compared in one session, alternating processes:
  for i in 1 2 3; do python tools/weighted_fit_cost.py --lib OLD.so; python tools/weighted_fit_cost.py; done
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np  # noqa: E402


def use_library(path):
    """Point the binding at another build; symbols that build lacks are left out of the binding."""
    from bore_b200 import _lib, build
    build.LIB_PATH = os.path.abspath(path)
    build.needs_build = lambda: False
    have = C.CDLL(build.LIB_PATH)
    for name in [n for n in _lib.SIGNATURES if not hasattr(have, n)]:
        del _lib.SIGNATURES[name]


def glorot(dims, rs):
    ws = []
    for fi, fo in zip(dims[:-1], dims[1:]):
        lim = np.sqrt(6.0 / (fi + fo))
        ws += [rs.uniform(-lim, lim, size=(fi, fo)).astype(np.float32), np.zeros(fo, np.float32)]
    return ws


def time_fit(dims, acts, M, N, E, mode, reps, weighted):
    import torch
    from bore_b200.engine import NativeMLP
    rs = np.random.RandomState(0)
    X = rs.uniform(size=(M * N, dims[0])).astype(np.float32)
    y = np.sum((X - 0.4) ** 2, axis=1).reshape(M, N)
    z = (y < np.quantile(y, 0.25, axis=1, keepdims=True)).astype(np.float32).reshape(-1)
    w = rs.uniform(0.0, 2.0, size=M * N).astype(np.float32)
    perm = np.stack([rs.permutation(N) for _ in range(E)]).astype(np.int32)
    net = NativeMLP(dims, acts, n_models=M)
    net.set_fit_mode(mode)
    w0 = glorot(dims, rs)
    for i in range(M):
        net.set_weights(w0, model=i)
    Xd, zd, pd = net.to_device(X, np.float32), net.to_device(z, np.float32), net.to_device(perm, np.int32)
    kw = dict(w_dev=net.to_device(w, np.float32), class_weight=(0.5, 2.0)) if weighted else {}
    times = []
    for r in range(reps + 1):
        net.reset_optimizer()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        net.fit_dev(Xd, zd, N, 64, E, pd, model0=0, count=M, shared_data=M == 1, shared_perm=True, **kw)
        e1.record()
        torch.cuda.synchronize()
        if r:
            times.append(e0.elapsed_time(e1))
    return min(times)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--lib", help="another build of libbore_b200.so to time")
    ap.add_argument("--reps", type=int, default=5)
    args = ap.parse_args()
    if args.lib:
        use_library(args.lib)
    from bore_b200 import _lib
    _lib.require_cuda()
    cfg3 = ([50, 64, 64, 64, 1], ["relu", "relu", "relu", "sigmoid"], 1, 2000, 31, 4)
    cfg4 = ([6, 32, 32, 1], ["relu", "relu", "sigmoid"], 4096, 500, 125, 1)
    out = {"lib": args.lib or "tree"}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30)
        out["gpu"] = q.stdout.strip().splitlines()[0]
    except (OSError, subprocess.SubprocessError, IndexError):
        out["gpu"] = "unknown"
    weighted = "bore_mlp_fit_weighted" in _lib.SIGNATURES
    for name, cfg in (("cfg3_mode4_ms", cfg3), ("cfg4_mode1_ms", cfg4)):
        out[name] = round(time_fit(*cfg, args.reps, False), 3)
        if weighted:
            out[name.replace("_ms", "_weighted_ms")] = round(time_fit(*cfg, args.reps, True), 3)
    print(json.dumps(out), flush=True)


if __name__ == "__main__":
    main()
