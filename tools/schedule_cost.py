"""What a learning-rate schedule costs in the fit kernels, and that the fits without one do not move.

Workloads (CUDA events, best of --reps after one warm-up each), as tools/regularizer_cost.py:
  fit_cfg3   one [50, 64, 64, 64, 1] relu model, N = 2,000, 31 epochs x 32 steps, fit mode 4 (unit-split K1u)
  fit_cfg4   4,096 [6, 32, 32, 1] relu models, N = 500 each, 125 epochs x 8 steps, fit mode 1 (one CTA each)
  lstm_fit   the multi-fidelity plugin's proposal fit: 2 x 32-unit tanh cells on 6 features, 4 rungs, N = 500,
             batch 64, 25 epochs x 8 steps
each under Adam and under RMSprop at a constant learning rate of 1e-3, and -- when the library has the schedule
setters -- under the same optimizers with ExponentialDecay(1e-3, 100, 0.9).  Adam with a schedule runs the OPT build
of every fit kernel, RMSprop runs it either way: the Adam pair shows the cost of that build, the RMSprop pair the
cost of evaluating the schedule.  Prints one JSON line with the device name and power limit; --out appends it to a
file.

--lib PATH times another build of libbore_b200.so (e.g. the parent commit's) through the same Python code;
alternate the two in one session to see the spread:
  for i in 1 2 3; do python tools/schedule_cost.py --lib OLD.so; python tools/schedule_cost.py; done
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
# case: (BORE_OPT_* kind, its BORE_OPT_NHP hyper-parameters, BORE_LR_* schedule and its parameters or None)
ADAM = (0, [1e-3, 0.9, 0.999, 1e-7, 0.0, 0.0, 0.0])
RMSPROP = (1, [1e-3, 0.9, 0.0, 1e-7, 0.0, 0.0, 0.0])
EXPONENTIAL = (1, [1e-3, 100.0, 0.9, 0.0])
CASES = {"adam": ADAM + (None,), "rmsprop": RMSPROP + (None,), "adam_exponential": ADAM + (EXPONENTIAL,),
         "rmsprop_exponential": RMSPROP + (EXPONENTIAL,)}


def _set(lib, h, case, mlp):
    """The case's optimizer through the C calls themselves: the schedule setter only where the case has a schedule,
    so that a build without it times the other cases."""
    from bore_b200 import _lib
    from bore_b200.engine import _np_ptr as np_ptr
    kind, hp, sched = CASES[case]
    pre = "bore_mlp_" if mlp else "bore_lstm_"
    _lib.check(getattr(lib, pre + "set_optimizer_kind")(h, kind, np_ptr(np.asarray(hp, np.float32))))
    if sched:
        sp = np.asarray(sched[1], np.float32)
        _lib.check(getattr(lib, pre + "set_lr_schedule")(h, sched[0], np_ptr(sp), sp.size))


def fit_case(dims, case, M, N, E, mode, reps):
    from bore_b200.engine import NativeMLP
    rs = np.random.RandomState(0)
    X = rs.uniform(size=(M * N, dims[0])).astype(np.float32)
    y = np.sum((X - 0.4) ** 2, axis=1).reshape(M, N)
    z = (y < np.quantile(y, 0.25, axis=1, keepdims=True)).astype(np.float32).reshape(-1)
    perm = np.stack([rs.permutation(N) for _ in range(E)]).astype(np.int32)
    net = NativeMLP(dims, ["relu"] * (len(dims) - 2) + ["sigmoid"], n_models=M)
    w = glorot(dims, np.random.RandomState(0))
    for i in range(M):
        net.set_weights(w, model=i)
    net.set_fit_mode(mode)
    _set(net.lib, net.h, case, True)
    Xd, zd, pd = net.to_device(X, np.float32), net.to_device(z, np.float32), net.to_device(perm, np.int32)

    def launch():
        net.reset_optimizer()
        net.fit_dev(Xd, zd, N, 64, E, pd, model0=0, count=M, shared_data=M == 1, shared_perm=True)
    return _time(launch, reps)


def lstm_case(case, reps):
    from bore_b200.recurrent import NativeLSTM
    D, U, L, T, N, E = 6, 32, 2, 4, 500, 25
    rs = np.random.RandomState(3)
    X = rs.uniform(size=(N, T, D)).astype(np.float32)
    Y = (rs.uniform(size=(N, T, 1)) < 0.4).astype(np.float32)
    perm = np.stack([rs.permutation(N) for _ in range(E)]).astype(np.int32)
    net = NativeLSTM(D, U, L, "tanh")
    net.set_weights([rs.uniform(-0.2, 0.2, size=s).astype(np.float32) for s in net.shapes()])
    _set(net.lib, net.h, case, False)
    return _time(lambda: net.fit_async(X, Y, E, 64, perm, -1.0), reps)


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
    runs = {
        "fit_cfg3": lambda c: fit_case(CFG3, c, 1, 2000, 31, 4, args.reps),
        "fit_cfg4": lambda c: fit_case(CFG4, c, 4096, 500, 125, 1, args.reps),
        "lstm_fit": lambda c: lstm_case(c, args.reps),
    }
    has_schedules = hasattr(lib, "bore_mlp_set_lr_schedule")
    for case in CASES:
        if CASES[case][2] and not has_schedules:
            continue
        for name, run in runs.items():
            out[f"{name}_{case}_ms"] = run(case)
    line = json.dumps(out)
    print(line, flush=True)
    if args.out:
        with open(args.out, "a") as fh:
            fh.write(line + "\n")


if __name__ == "__main__":
    main()
