"""What the activations selu, softplus, softsign, hard_sigmoid and exponential cost, and that the existing
nets do not move.

Workloads (CUDA events, best of --reps after one warm-up each):
  fit_cfg3   one [50, 64, 64, 64, 1] model, N = 2,000, 31 epochs x 32 steps, fit mode 4 (unit-split K1u)
  fit_cfg4   4,096 [6, 32, 32, 1] models, N = 500 each, 125 epochs x 8 steps, fit mode 1 (one CTA each)
  k2_cfg3    value and input gradient of the cfg-3 net at 65,536 points (K2)
  k3f_cfg2   fused L-BFGS-B argmax (K3f), 1,024 starts on the [6, 32, 32, 1] net
  k3f_cfg3   fused L-BFGS-B argmax (K3f), 4,096 starts on the cfg-3 net
each with the hidden activation relu (the benchmark's nets), elu, and -- when the library takes them -- every
new activation.  Prints one JSON line with the device name and power limit.

--lib PATH times another build of libbore_b200.so (e.g. the parent commit's) through the same Python code;
alternate the two in one session to see the spread:
  for i in 1 2 3; do python tools/activation_cost.py --lib OLD.so; python tools/activation_cost.py; done
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

from weighted_fit_cost import glorot, use_library  # noqa: E402

CFG3 = [50, 64, 64, 64, 1]
CFG2 = [6, 32, 32, 1]
ACTS = ("relu", "elu", "selu", "softplus", "softsign", "hard_sigmoid", "exponential")


def _time(launch, reps):
    import torch
    times = []
    for r in range(reps + 1):
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        launch()
        e1.record()
        torch.cuda.synchronize()
        if r:
            times.append(e0.elapsed_time(e1))
    return round(min(times), 3)


def _net(dims, act, M=1, head="sigmoid"):
    from bore_b200.engine import NativeMLP
    acts = [act] * (len(dims) - 2) + [head]
    net = NativeMLP(dims, acts, n_models=M)
    w = glorot(dims, np.random.RandomState(0))
    for i in range(M):
        net.set_weights(w, model=i)
    return net


def fit_case(dims, act, M, N, E, mode, reps):
    rs = np.random.RandomState(0)
    X = rs.uniform(size=(M * N, dims[0])).astype(np.float32)
    y = np.sum((X - 0.4) ** 2, axis=1).reshape(M, N)
    z = (y < np.quantile(y, 0.25, axis=1, keepdims=True)).astype(np.float32).reshape(-1)
    perm = np.stack([rs.permutation(N) for _ in range(E)]).astype(np.int32)
    net = _net(dims, act, M)
    net.set_fit_mode(mode)
    Xd, zd, pd = net.to_device(X, np.float32), net.to_device(z, np.float32), net.to_device(perm, np.int32)

    def launch():
        net.reset_optimizer()
        net.fit_dev(Xd, zd, N, 64, E, pd, model0=0, count=M, shared_data=M == 1, shared_perm=True)
    return _time(launch, reps)


def k2_case(act, reps):
    import torch
    net = _net(CFG3, act)
    X = torch.from_numpy(np.random.RandomState(1).uniform(size=(65536, 50)).astype(np.float32)).cuda()
    return _time(lambda: net.value_and_grad_dev(X, "identity", True), reps)


def k3f_case(dims, act, S, reps):
    import torch
    from bore_b200 import _lib
    net = _net(dims, act)
    X0 = torch.from_numpy(np.random.RandomState(2).uniform(size=(S, dims[0]))).cuda()
    lib = _lib.require_cuda()
    _lib.check(lib.bore_lbfgsb_set_mode(2))  # fused kernel only
    try:
        return _time(lambda: net.lbfgsb_dev(X0, 0.0, 1.0, transform="identity"), reps)
    finally:
        _lib.check(lib.bore_lbfgsb_set_mode(0))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--lib", help="another build of libbore_b200.so to time")
    ap.add_argument("--reps", type=int, default=5)
    args = ap.parse_args()
    if args.lib:
        use_library(args.lib)
    from bore_b200 import _lib
    from bore_b200._lib import BoreNativeError
    _lib.require_cuda()
    out = {"lib": args.lib or "tree"}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30)
        out["gpu"] = q.stdout.strip().splitlines()[0]
    except (OSError, subprocess.SubprocessError, IndexError):
        out["gpu"] = "unknown"
    cases = {
        "fit_cfg3": lambda a: fit_case(CFG3, a, 1, 2000, 31, 4, args.reps),
        "fit_cfg4": lambda a: fit_case(CFG2, a, 4096, 500, 125, 1, args.reps),
        "k2_cfg3": lambda a: k2_case(a, args.reps),
        "k3f_cfg2": lambda a: k3f_case(CFG2, a, 1024, args.reps),
        "k3f_cfg3": lambda a: k3f_case(CFG3, a, 4096, args.reps),
    }
    for act in ACTS:
        for name, run in cases.items():
            try:
                out[f"{name}_{act}_ms"] = run(act)
            except BoreNativeError:  # a build without this activation
                break
    print(json.dumps(out), flush=True)


if __name__ == "__main__":
    main()
