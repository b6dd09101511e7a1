"""What the optimizers RMSprop, Adagrad, Adadelta, Adamax and Nadam cost compared with Adam, and that Adam does
not move.

Workloads (CUDA events, best of --reps after one warm-up each):
  fit_cfg3   one [50, 64, 64, 64, 1] relu model, N = 2,000, 31 epochs x 32 steps, fit mode 4 (unit-split K1u)
  fit_cfg4   4,096 [6, 32, 32, 1] relu models, N = 500 each, 125 epochs x 8 steps, fit mode 1 (one CTA each)
  lstm_fit   the multi-fidelity plugin's proposal fit: 2 x 32-unit tanh cells on 6 features, 4 rungs, N = 500,
             batch 64, 25 epochs x 8 steps
each under Adam (the benchmark's optimizer) and -- when the library takes them -- every other kind, with Keras'
default hyper-parameters (RMSprop also with momentum 0.9 and centered).  Prints one JSON line with the device
name and power limit.

--lib PATH times another build of libbore_b200.so (e.g. the parent commit's) through the same Python code;
alternate the two in one session to see the spread:
  for i in 1 2 3; do python tools/optimizer_cost.py --lib OLD.so; python tools/optimizer_cost.py; done
"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.dirname(ROOT))
import numpy as np  # noqa: E402

from activation_cost import _time  # noqa: E402
from weighted_fit_cost import glorot, use_library  # noqa: E402

CFG3 = [50, 64, 64, 64, 1]
CFG4 = [6, 32, 32, 1]
KINDS = {
    "adam": None,  # the handle's own optimizer: no call the parent build lacks
    "rmsprop": dict(),
    "rmsprop_momentum": dict(momentum=0.9),
    "rmsprop_centered": dict(centered=True),
    "adagrad": dict(),
    "adadelta": dict(),
    "adamax": dict(),
    "nadam": dict(),
}


def _spec(kind):
    from bore_b200 import layers
    return type(layers.optimizer_spec(kind.split("_")[0]))(**KINDS[kind])


def fit_case(dims, kind, M, N, E, mode, reps):
    from bore_b200.engine import NativeMLP
    rs = np.random.RandomState(0)
    X = rs.uniform(size=(M * N, dims[0])).astype(np.float32)
    y = np.sum((X - 0.4) ** 2, axis=1).reshape(M, N)
    z = (y < np.quantile(y, 0.25, axis=1, keepdims=True)).astype(np.float32).reshape(-1)
    perm = np.stack([rs.permutation(N) for _ in range(E)]).astype(np.int32)
    net = NativeMLP(dims, ["relu"] * (len(dims) - 2) + ["sigmoid"], n_models=M)
    if KINDS[kind] is not None:
        net.set_optimizer_kind(_spec(kind))
    w = glorot(dims, np.random.RandomState(0))
    for i in range(M):
        net.set_weights(w, model=i)
    net.set_fit_mode(mode)
    Xd, zd, pd = net.to_device(X, np.float32), net.to_device(z, np.float32), net.to_device(perm, np.int32)

    def launch():
        net.reset_optimizer()
        net.fit_dev(Xd, zd, N, 64, E, pd, model0=0, count=M, shared_data=M == 1, shared_perm=True)
    return _time(launch, reps)


def lstm_case(kind, reps):
    from bore_b200.recurrent import NativeLSTM
    D, U, L, T, N, E = 6, 32, 2, 4, 500, 25
    rs = np.random.RandomState(3)
    X = rs.uniform(size=(N, T, D)).astype(np.float32)
    Y = (rs.uniform(size=(N, T, 1)) < 0.4).astype(np.float32)
    perm = np.stack([rs.permutation(N) for _ in range(E)]).astype(np.int32)
    net = NativeLSTM(D, U, L, "tanh")
    if KINDS[kind] is not None:
        net.set_optimizer_kind(_spec(kind))
    net.set_weights([rs.uniform(-0.2, 0.2, size=s).astype(np.float32) for s in net.shapes()])
    net.set_regularizers([0.0] * (3 * L + 2))
    return _time(lambda: net.fit_async(X, Y, E, 64, perm, -1.0), reps)


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
    cases = {
        "fit_cfg3": lambda k: fit_case(CFG3, k, 1, 2000, 31, 4, args.reps),
        "fit_cfg4": lambda k: fit_case(CFG4, k, 4096, 500, 125, 1, args.reps),
        "lstm_fit": lambda k: lstm_case(k, args.reps),
    }
    for kind in KINDS:
        for name, run in cases.items():
            try:
                out[f"{name}_{kind}_ms"] = run(kind)
            except AttributeError:  # a build without the optimizer kinds
                break
    print(json.dumps(out), flush=True)


if __name__ == "__main__":
    main()
