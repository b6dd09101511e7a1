"""What the lock-step L-BFGS-B stepper (lbfgsb_warp_kernel) costs on the benchmark's argmax.

Builds bench.py's cfg-3 model (Ackley-50, Dense64x3-ReLU + sigmoid, the same seeds), trains it once as
a bench step does, then runs the 65,536-start argmax --reps times after one warm-up call, with the
library's per-kernel timing on (bore_lbfgsb_profile).  Prints one JSON line: the device name and power
limit, stepper ms (the round kernels plus the fused tail they hand over to) and K2 ms per argmax (min,
median and max over the reps), the round count, and a digest of x / fun / nit / nfev / status / task:
two builds that compute the same bits print the same digest.

--lib PATH times another build of libbore_b200.so (e.g. the parent commit's) through the same Python
code, so that two builds can be compared in one session, alternating processes:
  for i in 1 2 3; do python tools/stepper_cost.py --lib OLD.so; python tools/stepper_cost.py; done
--handover N sets BORE_LB_HANDOVER (the active count at which the rounds hand over to the fused tail).
"""
import argparse
import ctypes as C
import hashlib
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.dirname(ROOT))
import numpy as np  # noqa: E402

from weighted_fit_cost import use_library  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--lib", help="another build of libbore_b200.so to time")
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--handover", type=int, help="BORE_LB_HANDOVER for this process")
    args = ap.parse_args()
    if args.handover is not None:
        os.environ["BORE_LB_HANDOVER"] = str(args.handover)
    if args.lib:
        use_library(args.lib)
    import torch
    import bench
    from bore_b200 import _lib, ops
    from bore_b200.layers import Dense
    from bore_b200.models import MaximizableSequential
    lib = _lib.require_cuda()
    out = {"lib": args.lib or "tree", "handover": os.environ.get("BORE_LB_HANDOVER", "default")}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30)
        out["gpu"] = q.stdout.strip().splitlines()[0]
    except (OSError, subprocess.SubprocessError, IndexError):
        out["gpu"] = "unknown"

    # bench.py's cfg-3 step, rank 0: the same problem, initial weights, fit and start points
    wl = bench.WORKLOADS["cfg3"]
    dims, acts, D, S = wl["dims"], wl["acts"], wl["dims"][0], wl["starts"]
    X, z, perms = bench.make_problem(wl, seed=0)
    model = MaximizableSequential(transform=ops.TRANSFORMS[wl["transform"]], device=0)
    for i, (u, a) in enumerate(zip(dims[1:], acts)):
        model.add(Dense(u, activation=a, input_dim=D if i == 0 else None))
    model.compile(optimizer="adam", loss="binary_crossentropy")
    model.set_weights(bench.glorot_init(dims, 0))
    net = model._engine(D)
    net.fit_dev(net.to_device(X, np.float32), net.to_device(z.astype(np.float32), np.float32), wl["N"],
                wl["batch"], wl["epochs"], net.to_device(perms, np.int32))
    X0d = net.to_device(np.random.RandomState(1000).uniform(size=(S, D)), np.float64)
    lo, hi = np.zeros(D), np.ones(D)
    opts = dict(m=10, ftol=1e-9, gtol=1e-5, maxiter=1000, maxfun=15000, maxls=20)
    tname = model._min_transform_name()

    prof = np.zeros(8)
    step, k2, rounds, digest = [], [], set(), set()
    for r in range(args.reps + 1):
        torch.cuda.synchronize()
        lib.bore_lbfgsb_profile(1)
        res = net.lbfgsb_dev(X0d, lo, hi, transform=tname, **opts)
        torch.cuda.synchronize()
        lib.bore_lbfgsb_profile(0)
        lib.bore_lbfgsb_last_profile(prof.ctypes.data_as(C.POINTER(C.c_double)))
        h = hashlib.sha256()
        for k in ("x", "fun", "nit", "nfev", "status", "task"):
            h.update(res[k].cpu().numpy().tobytes())
        digest.add(h.hexdigest()[:16])
        if r:  # the first call is the warm-up
            step.append(prof[1])
            k2.append(prof[0])
            rounds.add(int(prof[2]))
    if prof[5]:
        out["warning"] = "the argmax ran the fused persistent kernel, not the rounds"
    stat = lambda v: [round(min(v), 3), round(float(np.median(v)), 3), round(max(v), 3)]
    out["stepper_ms_min_med_max"] = stat(step)
    out["k2_ms_min_med_max"] = stat(k2)
    out["rounds"] = sorted(rounds)
    out["digest"] = sorted(digest)
    print(json.dumps(out), flush=True)


if __name__ == "__main__":
    main()
