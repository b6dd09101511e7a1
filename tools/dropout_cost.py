"""What Dropout costs in the MLP fit kernels, and that the fits without it do not move.

Workloads (CUDA events, best of --reps after one warm-up each), as tools/schedule_cost.py:
  fit_cfg3   one [50, 64, 64, 64, 1] relu model, N = 2,000, 31 epochs x 32 steps, fit mode 4 (unit-split K1u)
  fit_cfg4   4,096 [6, 32, 32, 1] relu models, N = 500 each, 125 epochs x 8 steps, fit mode 1 (one CTA each)
  fit_cfg5   one [8, 32, 32, 32, 1] elu model (the plugin's net), N = 500, 125 epochs x 8 steps, automatic fit mode
each under Adam and under RMSprop, without dropout and -- when the library has bore_mlp_set_dropout -- with
Dropout(0.2) after every hidden layer.  Dropout runs the OPT build of every fit kernel, RMSprop runs it either way: the
Adam pair shows the cost of that build plus the masks, the RMSprop pair the cost of the masks alone.  Prints one JSON
line with the device name and power limit; --out appends it to a file.

--lib PATH times another build of libbore_b200.so (e.g. the parent commit's) through the same Python code;
alternate the two in one session to see the spread:
  for i in 1 2 3; do python tools/dropout_cost.py --lib OLD.so; python tools/dropout_cost.py; done
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

# case: (BORE_OPT_* kind, its BORE_OPT_NHP hyper-parameters, dropout rate after every hidden layer)
ADAM = (0, [1e-3, 0.9, 0.999, 1e-7, 0.0, 0.0, 0.0])
RMSPROP = (1, [1e-3, 0.9, 0.0, 1e-7, 0.0, 0.0, 0.0])
CASES = {"adam": ADAM + (0.0,), "rmsprop": RMSPROP + (0.0,), "adam_dropout": ADAM + (0.2,),
         "rmsprop_dropout": RMSPROP + (0.2,)}
# workload: (dims, hidden activation, models, N, epochs, fit mode)
FITS = {"fit_cfg3": ([50, 64, 64, 64, 1], "relu", 1, 2000, 31, 4),
        "fit_cfg4": ([6, 32, 32, 1], "relu", 4096, 500, 125, 1),
        "fit_cfg5": ([8, 32, 32, 32, 1], "elu", 1, 500, 125, 0)}


def fit_case(fit, case, reps):
    from bore_b200 import _lib
    from bore_b200.engine import NativeMLP, _np_ptr
    dims, act, M, N, E, mode = FITS[fit]
    kind, hp, rate = CASES[case]
    rs = np.random.RandomState(0)
    X = rs.uniform(size=(M * N, dims[0])).astype(np.float32)
    y = np.sum((X - 0.4) ** 2, axis=1).reshape(M, N)
    z = (y < np.quantile(y, 0.25, axis=1, keepdims=True)).astype(np.float32).reshape(-1)
    perm = np.stack([rs.permutation(N) for _ in range(E)]).astype(np.int32)
    net = NativeMLP(dims, [act] * (len(dims) - 2) + ["sigmoid"], n_models=M)
    w = glorot(dims, np.random.RandomState(0))
    for i in range(M):
        net.set_weights(w, model=i)
    net.set_fit_mode(mode)
    _lib.check(net.lib.bore_mlp_set_optimizer_kind(net.h, kind, _np_ptr(np.asarray(hp, np.float32))))
    if rate > 0:  # through the C call itself, so that a build without it times the other cases
        n = len(dims) - 2
        r, s = np.full(n, rate, np.float32), np.arange(1, n + 1, dtype=np.uint32)
        _lib.check(net.lib.bore_mlp_set_dropout(net.h, n, _np_ptr(r), _np_ptr(s)))
    Xd, zd, pd = net.to_device(X, np.float32), net.to_device(z, np.float32), net.to_device(perm, np.int32)

    def launch():
        net.reset_optimizer()
        net.fit_dev(Xd, zd, N, 64, E, pd, model0=0, count=M, shared_data=M == 1, shared_perm=True)
    return _time(launch, reps)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--lib", help="another build of libbore_b200.so to time")
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", help="append the JSON line to this file too")
    args = ap.parse_args()
    if args.lib:
        use_library(args.lib)
    from bore_b200 import _lib
    _lib.require_cuda()
    lib = _lib.load()
    out = {"lib": "other" if args.lib else "tree"}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30)
        out["gpu"] = q.stdout.strip().splitlines()[0]
    except (OSError, subprocess.SubprocessError, IndexError):
        out["gpu"] = "unknown"
    has_dropout = hasattr(lib, "bore_mlp_set_dropout")
    for case in CASES:
        if CASES[case][2] > 0 and not has_dropout:
            continue
        for fit in FITS:
            out[f"{fit}_{case}_ms"] = fit_case(fit, case, args.reps)
    line = json.dumps(out)
    print(line, flush=True)
    if args.out:
        with open(args.out, "a") as fh:
            fh.write(line + "\n")


if __name__ == "__main__":
    main()
