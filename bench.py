#!/usr/bin/env python
"""bench.py -- the BORE-MLP hot path (fit -> multi-start argmax) on N B200s.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload cfg3]
                    [--dump-outputs DIR]

A "step" is one BO iteration on synthetic quantile-labelled data: fit the classifier (Keras
semantics: `epochs` x ceil(N/64) Adam steps) then maximise it from S start points with the
batched on-device L-BFGS-B.  Default workload = BASELINE.json configs[2], the configuration
north_star's target is quoted on: synthetic 50-D Ackley, Dense64 x3 (+ sigmoid output), 2,000
observations, 65,536 starts per GPU.  Multi-GPU is WEAK scaling: weights replicated (every rank
runs the same deterministic fit), every rank optimises its own 65,536 starts, one NCCL max
all-reduce on the packed (value, index) key picks the global argmax.  The same JSON line carries
two sub-records: `strong` (the SAME 65,536 starts in total split over the N ranks, 3 steps --
north_star's "fit + 65,536-start argmax" from 1 to 8 GPUs) and `cfg4` (BASELINE.json configs[3]:
4,096 independent BO problems split over the ranks, 2 steps).

`value` = value+input-gradient evaluations per second, whole job, inputs resident in HBM,
timed with CUDA events (max over ranks).  `e2e` = the same through the public Python API
(`model.fit` / `model.argmax`) with HOST numpy buffers, copies inside the timed region.
`roofline` describes the kernel with the largest share of the step, `kernels` all of them.
`cpu_baseline` (N=1 only) and `--impl reference` time the oracle's restatement of the reference's
CPU path (NumPy Keras semantics + one scipy.optimize.minimize per start) -- TensorFlow cannot be
installed in this image, see DESIGN.md -- on the box's host cores.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

WORKLOADS = {
    # BASELINE.json configs[2]
    "cfg3": dict(name="Ackley-50 / Dense64x3-ReLU+sigmoid / N=2000 / 65536 starts per GPU",
                 dims=[50, 64, 64, 64, 1], acts=["relu", "relu", "relu", "sigmoid"],
                 transform="identity", N=2000, epochs=31, batch=64, starts=65536, gamma=0.25,
                 target="ackley"),
    # BASELINE.json configs[1]
    "cfg2": dict(name="Hartmann-6 / Dense32x2-ReLU+sigmoid / N=500 / 1024 starts",
                 dims=[6, 32, 32, 1], acts=["relu", "relu", "sigmoid"], transform="identity",
                 N=500, epochs=125, batch=64, starts=1024, gamma=0.25, target="hartmann6"),
    # plugin defaults (BASELINE.json configs[4] network)
    "cfg5": dict(name="8-D plugin net / Dense32x3-ELU logits + sigmoid transform / N=500 / 65536 starts",
                 dims=[8, 32, 32, 32, 1], acts=["elu", "elu", "elu", "linear"], transform="sigmoid",
                 N=500, epochs=125, batch=64, starts=65536, gamma=1 / 3, target="ackley"),
}

NOMINAL_FP32_TFLOPS = 148 * 128 * 2 * 1.965e9 / 1e12  # 74.4


def ackley(X):
    u = -32.768 + 65.536 * X
    d = X.shape[1]
    return (-20.0 * np.exp(-0.2 * np.sqrt(np.sum(u * u, axis=1) / d))
            - np.exp(np.sum(np.cos(2 * np.pi * u), axis=1) / d) + 20.0 + np.e)


_H_A = np.array([[10, 3, 17, 3.5, 1.7, 8], [0.05, 10, 17, 0.1, 8, 14], [3, 3.5, 1.7, 10, 17, 8],
                 [17, 8, 0.05, 10, 0.1, 14]])
_H_P = 1e-4 * np.array([[1312, 1696, 5569, 124, 8283, 5886], [2329, 4135, 8307, 3736, 1004, 9991],
                        [2348, 1451, 3522, 2883, 3047, 6650], [4047, 8828, 8732, 5743, 1091, 381]])


def hartmann6(X):
    al = np.array([1.0, 1.2, 3.0, 3.2])
    inner = np.einsum("ij,nij->ni", _H_A, (X[:, None, :] - _H_P[None]) ** 2)
    return -np.sum(al * np.exp(-inner), axis=1)


def make_problem(wl, seed):
    rs = np.random.RandomState(seed)
    D = wl["dims"][0]
    X = rs.uniform(size=(wl["N"], D))
    y = {"ackley": ackley, "hartmann6": hartmann6}[wl["target"]](X)
    z = y < np.quantile(y, wl["gamma"])
    perms = np.stack([rs.permutation(wl["N"]) for _ in range(wl["epochs"])]).astype(np.int32)
    return X, z, perms


def glorot_init(dims, seed):
    """Keras-ordered weights [W0 (in,out), b0, W1, b1, ...]: glorot_uniform kernels from
    RandomState(seed), zero biases -- the synthetic random-init weights of both arms (spelled out here
    so that the GPU arm imports nothing from oracle/)."""
    rs = np.random.RandomState(seed)
    ws = []
    for fi, fo in zip(dims[:-1], dims[1:]):
        lim = np.sqrt(6.0 / (fi + fo))
        ws.append(rs.uniform(-lim, lim, size=(fi, fo)).astype(np.float32))
        ws.append(np.zeros(fo, np.float32))
    return ws


def workload_config(wl):
    """The `config` object of the JSON line -- the SAME dict for both arms (--impl ours / reference);
    anything descriptive goes under `notes`."""
    return {"workload": wl["name"], "starts_per_gpu": wl["starts"], "observations": wl["N"],
            "adam_steps": wl["epochs"] * (-(-wl["N"] // wl["batch"]))}


def flops_per_eval(dims):
    return 4 * sum(a * b for a, b in zip(dims[:-1], dims[1:]))


def flops_per_fit_step(dims, batch):
    W = sum(a * b for a, b in zip(dims[:-1], dims[1:]))
    P = W + sum(dims[1:])
    return batch * (6 * W - 2 * dims[0] * dims[1]) + 12 * P


# ------------------------------------------------------------------------------ clocks
class ClockSampler:
    QUERY = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
             "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu, self.proc, self.lines = gpu_index, None, []

    def start(self):
        if self.gpu is None:  # ranks other than 0 do not sample: N nvidia-smi loops on one box take turns at a
            return            # driver-wide lock and stall each other's kernel launches (8 ranks: +16 ms per step)
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu),
                                          "--query-gpu=" + self.QUERY, "--format=csv,noheader,nounits",
                                          "-lms", "100"], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.proc is None:
            return dict(sm_mhz=None, sm_max_mhz=None, reasons=["nvidia-smi unavailable"])
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, smax, reasons, power = [], [], set(), []
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            f = [t.strip() for t in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); smax.append(float(f[2])); power.append(float(f[3]))
            except ValueError:
                continue
            for nm, v in zip(names, f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        if not sm:
            return dict(sm_mhz=None, sm_max_mhz=None, reasons=["no samples"])
        return dict(sm_mhz=float(np.median(sm)), sm_max_mhz=float(max(smax)),
                    reasons=sorted(reasons), samples=len(sm), power_w_max=float(max(power)))


# ------------------------------------------------------------------------------ reference arm
def _ref_worker(args):
    weights, acts, transform, X0 = args
    from scipy.optimize import Bounds
    from threadpoolctl import threadpool_limits
    from oracle import argmax as am
    n = X0.shape[1]
    with threadpool_limits(1):  # batch-of-1 matmuls: BLAS threading only adds contention
        r = am.minimize_starts(weights, acts, X0, Bounds(np.zeros(n), np.ones(n)), transform=transform)
    return int(r["nfev"].sum()), float(r["fun"].min())


def reference_step(wl, X, z, perms, w0, X0, pool, cores):
    """One bounded-sample step of the restated reference CPU path.  Returns (fit_s, argmax_s,
    evals in the sample)."""
    from oracle import keras_mlp as km
    from threadpoolctl import threadpool_limits
    w = [a.copy() for a in w0]
    t0 = time.perf_counter()
    with threadpool_limits(1):
        km.fit(w, wl["acts"], X, z, wl["epochs"], wl["batch"], perms)
    t1 = time.perf_counter()
    chunks = np.array_split(X0, cores)
    jobs = [(w, wl["acts"], wl["transform"], c) for c in chunks if len(c)]
    if pool is None:
        outs = [_ref_worker(j) for j in jobs]
    else:
        outs = pool.map(_ref_worker, jobs)
    t2 = time.perf_counter()
    return t1 - t0, t2 - t1, sum(o[0] for o in outs)


def run_reference(args, wl, rank, world):
    if rank != 0:
        return
    import multiprocessing as mp
    from oracle import keras_mlp as km
    cores = os.cpu_count() or 1
    X, z, perms = make_problem(wl, seed=0)
    w0 = km.init_weights(wl["dims"], 0)
    S_ref = min(wl["starts"], 64 * cores)
    X0 = np.random.RandomState(1).uniform(size=(S_ref, wl["dims"][0]))
    pool = None
    if cores > 1:
        # forked workers (NumPy / SciPy only): collect and freeze the parent's objects first so that a
        # child's garbage collector never runs a destructor that touches CUDA (tests/helpers.py::fork_pool)
        import gc
        gc.collect()
        gc.freeze()
        try:
            pool = mp.get_context("fork").Pool(cores)
        finally:
            gc.unfreeze()
    for _ in range(args.warmup):
        reference_step(wl, X, z, perms, w0, X0[:cores * 4], pool, cores)
    tf = ta = 0.0
    ev = 0
    for _ in range(args.steps):
        a, b, c = reference_step(wl, X, z, perms, w0, X0, pool, cores)
        tf += a; ta += b; ev += c
    if pool is not None:
        pool.close()
    K = args.steps
    scale = wl["starts"] / S_ref
    full_step_s = tf / K + (ta / K) * scale          # linear in the number of starts
    evals_full = ev / K * scale
    value = evals_full / full_step_s
    line = {
        "impl": "reference", "metric": "mlp_value_and_input_grad_evals_per_sec", "value": value,
        "unit": "evals/s", "n_gpus": args.gpus, "steps": K, "warmup": args.warmup,
        "ms_per_step": 1e3 * (tf + ta) / K, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32 MLP / f64 L-BFGS-B", "data": "synthetic",
        "config": workload_config(wl),
        "cpu_baseline": {"value": value, "unit": "evals/s", "cores": cores, "kind": "port",
                         "sample": f"full fit ({wl['epochs']} epochs, serial) + {S_ref} of "
                                   f"{wl['starts']} starts spread over {cores} processes per step; "
                                   "value extrapolated linearly in the number of starts; NumPy "
                                   "restatement of Keras + the installed SciPy L-BFGS-B, not TF"},
        "e2e": {"value": value, "unit": "evals/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "bo_iterations_per_sec": 1.0 / full_step_s,
        "phases": {"fit_ms": 1e3 * tf / K, "argmax_sample_ms": 1e3 * ta / K},
    }
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------ our arm
def run_ours(args, wl, rank, local_rank, world):
    import ctypes as C
    import torch
    import torch.distributed as dist
    from bore_b200 import ops, _lib
    from bore_b200.engine import ffma_peak_tflops
    from bore_b200.layers import Dense
    from bore_b200.models import MaximizableSequential
    from bore_b200 import distributed as bd

    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    lib = _lib.require_cuda()
    dims, acts, D, S = wl["dims"], wl["acts"], wl["dims"][0], wl["starts"]
    X, z, perms = make_problem(wl, seed=0)              # the same problem on every rank
    w0 = glorot_init(dims, 0)
    model = MaximizableSequential(transform=ops.TRANSFORMS[wl["transform"]], device=local_rank)
    for i, (u, a) in enumerate(zip(dims[1:], acts)):
        model.add(Dense(u, activation=a, input_dim=D if i == 0 else None))
    model.compile(optimizer="adam", loss="binary_crossentropy" if acts[-1] == "sigmoid" else
                  __import__("bore_b200").BinaryCrossentropy(from_logits=True))
    model.set_weights(w0)
    net = model._engine(D)
    bounds = [(0.0, 1.0)] * D
    lo, hi = np.zeros(D), np.ones(D)
    tname = model._min_transform_name()

    # ---- resident inputs (this rank's shard of the start points: its own seed) ----
    Xd = net.to_device(X, np.float32)
    zd = net.to_device(z.astype(np.float32), np.float32)
    pd = net.to_device(perms, np.int32)
    X0 = np.random.RandomState(1000 + rank).uniform(size=(S, D))
    X0d = net.to_device(X0, np.float64)
    X0f = X0d.to(torch.float32)
    params = net.params_tensor()
    w0d = params.clone()
    loss_d = torch.empty(1, wl["epochs"], dtype=torch.float32, device=dev)
    opts = dict(m=10, ftol=1e-9, gtol=1e-5, maxiter=1000, maxfun=15000, maxls=20)
    prof = np.zeros(8)

    def reset_state():
        params.copy_(w0d)
        net.reset_optimizer()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def make_step(X0d_, X0f_, S_local, idx_offset, S_total):
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(3)]
        zbuf = torch.empty(S_local, dtype=torch.float32, device=dev)

        def step(timers=None):
            """fit -> screening predict -> batched L-BFGS-B -> first-minimum key (-> NCCL max)."""
            reset_state()                                      # same work every step (see notes)
            if timers is not None:
                ev[0].record()
            net.fit_dev(Xd, zd, wl["N"], wl["batch"], wl["epochs"], pd, loss_dev=loss_d)
            if timers is not None:
                ev[1].record()
            net.predict_dev(X0f_, zbuf)                         # maxima's screening pass (mixins.py:50)
            res = net.lbfgsb_dev(X0d_, lo, hi, transform=tname, **opts)
            key = net.select_best(res["fun"], res["status"], idx_offset=idx_offset)
            rec_fn = lambda i: torch.cat([res["x"][i], res["fun"][i:i + 1]])
            gidx, rec = bd.global_winner(key, rec_fn, S_total, D + 1)
            if timers is not None:
                ev[2].record()
                torch.cuda.synchronize()
                timers["fit_ms"] += ev[0].elapsed_time(ev[1])
                timers["argmax_ms"] += ev[1].elapsed_time(ev[2])
            return res, gidx, rec, zbuf
        return step

    def timed(step, K, warm):
        """EXACTLY K steps between barrier + synchronize, CUDA events, max over ranks.  Also returns what
        the last step returned."""
        for _ in range(warm):
            step()
        agg = dict(k2_ms=0.0, step_ms=0.0, rounds=0, bytes=0.0, evals=0.0, fused=0, grid=0, block=0)
        timers = dict(fit_ms=0.0, argmax_ms=0.0)
        lib.bore_lbfgsb_profile(1)
        total_evals = 0
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(K):
            t_dbg = time.perf_counter()
            last = step(timers)
            res = last[0]
            if os.environ.get("BENCH_DEBUG"):
                sys.stderr.write(f"step {1e3 * (time.perf_counter() - t_dbg):.1f} ms rounds {res['rounds']} evals {res['evals']}\n")
            total_evals += res["evals"]
            lib.bore_lbfgsb_last_profile(prof.ctypes.data_as(C.POINTER(C.c_double)))
            agg["k2_ms"] += prof[0]; agg["step_ms"] += prof[1]; agg["rounds"] += int(prof[2])
            agg["bytes"] += prof[3]; agg["evals"] += prof[4]
            agg["fused"], agg["grid"], agg["block"] = int(prof[5]), int(prof[6]), int(prof[7])
        e1.record()
        barrier()
        lib.bore_lbfgsb_profile(0)
        elapsed_ms = e0.elapsed_time(e1)
        t = torch.tensor([elapsed_ms, float(total_evals)], dtype=torch.float64, device=dev)
        if world > 1:
            tmax = t.clone(); dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
            tsum = t.clone(); dist.all_reduce(tsum, op=dist.ReduceOp.SUM)
            elapsed_ms, evals_all = tmax[0].item(), tsum[1].item()
        else:
            evals_all = float(total_evals)
        return elapsed_ms, evals_all, agg, timers, last

    peak_ffma = ffma_peak_tflops(local_rank)
    peaks = {}
    mp_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(mp_path):
        peaks = json.load(open(mp_path))
    hbm_peak = float(peaks.get("hbm_gbs", 6650.0))
    hbm_src = "MEASURED_PEAKS.json hbm_gbs (of measured)" if peaks else "6650 GB/s (of fallback)"

    # ---- inputs of the strong-scaling record first: no host work (and no idle GPU) between the two timed parts ----
    Ks = 3
    lo_s, hi_s = bd.shard_bounds(S, rank, world)
    X0g = np.random.RandomState(1).uniform(size=(S, D))[lo_s:hi_s]   # same draw everywhere, own slice
    X0gd = net.to_device(np.ascontiguousarray(X0g), np.float64)
    step_strong = make_step(X0gd, X0gd.to(torch.float32), hi_s - lo_s, lo_s, S)

    # ---- headline: weak scaling, 65,536 starts on every GPU ----
    K, W = args.steps, max(args.warmup, 3)
    step_weak = make_step(X0d, X0f, S, rank * S, S * world)
    sampler = ClockSampler(local_rank if rank == 0 else None)
    sampler.start()  # before the warm-up: nvidia-smi starting up (NVML init) stalls launches -- one step of 198 ms
                     # instead of 125 when it was started right in front of the timed steps
    for _ in range(W):
        t_w = time.perf_counter()
        step_weak()
        if os.environ.get("BENCH_DEBUG"):
            torch.cuda.synchronize()
            sys.stderr.write(f"warm-up step {1e3 * (time.perf_counter() - t_w):.1f} ms\n")
    elapsed_ms, evals_all, agg, timers, last = timed(step_weak, K, 0)
    ms_per_step = elapsed_ms / K
    value = evals_all / (elapsed_ms * 1e-3)
    outputs = None
    if args.dump_outputs:
        # the next step resets the parameters in place: copy them (and the loss buffer) now, on the device
        res, gidx, rec, screen = last
        outputs = dict(fit_params=params.clone(), fit_loss=loss_d.clone(), screen_pred=screen,
                       **{"argmax_" + k: res[k] for k in ("x", "fun", "nit", "nfev", "status", "task")},
                       winner_index=np.array([-1 if gidx is None else gidx]),
                       winner_x_fun=np.full(D + 1, np.nan) if rec is None else rec)
    del last

    # ---- strong scaling: the SAME 65,536 starts in total, split over the ranks ----
    # (right behind the headline steps: measured after the 0.3 s of host work and idle GPU that used to sit
    #  here, the same three steps took anything from 131 to 205 ms on one GPU, where they ARE the headline step)
    s_ms, s_evals, s_agg, s_tim, _ = timed(step_strong, Ks, 3)
    clocks = sampler.stop()

    # ---- e2e: the public API with HOST buffers (H2D/D2H inside the timed region) ----
    rs = np.random.RandomState(2000 + rank)
    e2e_steps = max(2, min(K, 3))
    reset_state()
    zeros = [np.zeros_like(a) for a in w0]

    def api_step():
        # the same work as a resident step: start from the same weights and a fresh optimizer
        model.set_weights(w0)
        model.set_optimizer_state(zeros, zeros, 0)
        model.fit(X, z, epochs=wl["epochs"], batch_size=wl["batch"], verbose=0, permutations=perms)
        if world > 1:
            return model.argmax_sharded(bounds, num_starts=S, random_state=rs)
        return model.argmax(bounds, num_starts=S, num_samples=S, print_fn=None, random_state=rs)
    api_step()  # warm
    barrier()
    t0 = time.perf_counter()
    e2e_evals = 0
    for _ in range(e2e_steps):
        api_step()
        e2e_evals += model._last_stats["evals"]
    barrier()
    e2e_s = time.perf_counter() - t0
    te = torch.tensor([e2e_s, float(e2e_evals)], dtype=torch.float64, device=dev)
    if world > 1:
        a = te.clone(); dist.all_reduce(a, op=dist.ReduceOp.MAX)
        b = te.clone(); dist.all_reduce(b, op=dist.ReduceOp.SUM)
        e2e_s, e2e_evals = a[0].item(), b[1].item()
    n_par = sum(a.size for a in w0)
    h2d = X.size * 4 + z.size * 4 + perms.size * 4 + S * D * 8 + 3 * n_par * 4
    d2h = wl["epochs"] * 4 + (D + 5) * 8 + 8

    # ---- cfg 4 (BASELINE.json configs[3]) in short: 4,096 problems split over the ranks ----
    del X0d, X0f, X0gd
    cfg4 = None
    if not args.no_cfg4:
        cfg4 = cfg4_measure(rank, local_rank, world, steps=2, warm=1)
    if outputs is not None:
        write_outputs(args.dump_outputs, outputs, f"_rank{rank}" if world > 1 else "")

    if rank != 0:
        return
    # ---- per-kernel accounting over the timed region (CUDA events on the launch stream) ----
    F_eval = flops_per_eval(dims)
    n_adam = wl["epochs"] * (-(-wl["N"] // wl["batch"]))
    tot = timers["fit_ms"] + timers["argmax_ms"]
    fit_tflops = K * n_adam * flops_per_fit_step(dims, wl["batch"]) / (timers["fit_ms"] * 1e-3) / 1e12
    opt_ms = agg["k2_ms"] + agg["step_ms"]                     # K2 + stepper (or the fused kernel)
    opt_tflops = agg["evals"] * F_eval / (opt_ms * 1e-3) / 1e12
    step_gbs = agg["bytes"] / (agg["step_ms"] * 1e-3) / 1e9
    ffma_src = "FFMA microbenchmark measured in this run (nominal %.1f)" % NOMINAL_FP32_TFLOPS
    kernels = []
    if agg["fused"]:
        kernels.append(dict(name="lbfgsb_fused_kernel (K3f: persistent L-BFGS-B with the MLP inlined)",
                            bound="latency", ms_per_step=agg["step_ms"] / K, share=agg["step_ms"] / tot,
                            launches_per_step=1, achieved=opt_tflops, peak=peak_ffma, unit="TFLOP/s",
                            frac=opt_tflops / peak_ffma, peak_source=ffma_src,
                            hbm=dict(achieved=step_gbs, peak=hbm_peak, unit="GB/s", frac=step_gbs / hbm_peak)))
    else:
        k2_tflops = agg["evals"] * F_eval / (agg["k2_ms"] * 1e-3) / 1e12
        kernels.append(dict(name="lbfgsb_warp_kernel (K3 stepper)", bound="latency", ms_per_step=agg["step_ms"] / K,
                            share=agg["step_ms"] / tot, launches_per_step=agg["rounds"] / K, achieved=step_gbs,
                            peak=hbm_peak, unit="GB/s", frac=step_gbs / hbm_peak, peak_source=hbm_src))
        kernels.append(dict(name="mlp_eval_kernel<grad> (K2 value+input-grad)", bound="fp32_ffma",
                            ms_per_step=agg["k2_ms"] / K, share=agg["k2_ms"] / tot,
                            launches_per_step=agg["rounds"] / K, achieved=k2_tflops, peak=peak_ffma,
                            unit="TFLOP/s", frac=k2_tflops / peak_ffma, peak_source=ffma_src,
                            frac_of_nominal=k2_tflops / NOMINAL_FP32_TFLOPS))
    kernels.append(dict(name="fit_unit_kernel (K1u fused training, 1 model = one 8-CTA cluster, hidden units split over the CTAs)",
                        bound="latency (8 SMs)", ms_per_step=timers["fit_ms"] / K, share=timers["fit_ms"] / tot,
                        launches_per_step=1, achieved=fit_tflops, peak=peak_ffma * 8 / 148, unit="TFLOP/s",
                        frac=fit_tflops / (peak_ffma * 8 / 148), peak_source="8 SMs' share of the FFMA peak"))
    dom = kernels[0]
    # The dominant kernel is LATENCY bound (ncu: issue slots ~35 % busy, HBM < 16 % busy, fp64 pipe
    # < 10 %), so neither roofline binds; both fractions are reported: `frac` against the HBM byte
    # model of the kernel (DESIGN.md) and `fp32` = sum(nfev) * 4W FLOP over the K2 + K3 time against
    # the FFMA peak, the roofline SURVEY.md 8(d) names for the argmax.  `traffic` is null: it is not
    # measured inside this run (the ncu captures under profiles/ hold dram bytes per launch).
    roofline = dict(kernel=dom["name"], bound="latency",
                    achieved=step_gbs, peak=hbm_peak, unit="GB/s", frac=step_gbs / hbm_peak,
                    peak_source=hbm_src, traffic=None,
                    fp32=dict(achieved=opt_tflops, peak=peak_ffma, unit="TFLOP/s", frac=opt_tflops / peak_ffma,
                              peak_source=ffma_src, over="K2 + K3 time of the argmax",
                              frac_over_whole_step=(agg["evals"] * F_eval / (tot * 1e-3) / 1e12) / peak_ffma),
                    share_of_step=dom["share"], launches_per_step=dom["launches_per_step"])
    strong = {"scaling": "strong", "n_gpus": world, "steps": Ks, "total_starts": S,
              "starts_per_gpu": hi_s - lo_s, "ms_per_step": s_ms / Ks,
              "value": s_evals / (s_ms * 1e-3), "unit": "evals/s",
              "bo_iterations_per_sec": 1e3 / (s_ms / Ks),
              "phases": {"fit_ms": s_tim["fit_ms"] / Ks, "argmax_ms": s_tim["argmax_ms"] / Ks},
              "argmax_path": "fused persistent kernel" if s_agg["fused"] else "lock-step rounds",
              "note": "fit is replicated on every rank (weights replicated), so it is the Amdahl term: "
                      "speed-up <= (fit + argmax) / (fit + argmax / N)"}
    line = {
        "metric": "mlp_value_and_input_grad_evals_per_sec", "value": value, "unit": "evals/s",
        "n_gpus": world, "steps": K, "warmup": W, "ms_per_step": ms_per_step,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32 MLP / f64 L-BFGS-B", "data": "synthetic",
        "config": workload_config(wl),
        "notes": {"parallelism": f"starts sharded x{world}, weights replicated",
                  "l2_cache": "inputs larger than L2: per-start L-BFGS-B state %.2f GB per GPU streams "
                              "through HBM every round (>> 126 MB L2); no explicit flush" %
                              (S * (256 + (4 * D + D * 21 + 500) * 8) / 1e9),
                  "step": "weights and Adam state reset to the same seed before every step",
                  "argmax_path": "fused persistent kernel" if agg["fused"] else "lock-step rounds"},
        "bo_iterations_per_sec": 1e3 / ms_per_step,
        "phases": {"fit_ms": timers["fit_ms"] / K, "argmax_ms": timers["argmax_ms"] / K,
                   "lbfgsb_rounds": agg["rounds"] / K, "evals_per_step_per_gpu": agg["evals"] / K,
                   "argmax_evals_per_sec": world * agg["evals"] / (timers["argmax_ms"] * 1e-3)},
        "roofline": roofline, "kernels": kernels,
        "e2e": {"value": e2e_evals / e2e_s, "unit": "evals/s", "h2d_bytes_per_step": int(h2d),
                "d2h_bytes_per_step": int(d2h), "ms_per_step": 1e3 * e2e_s / e2e_steps,
                "steps": e2e_steps, "api": "MaximizableSequential.fit + .argmax (numpy in/out)"},
        # per step: reset (2 copies are not kernels) + fit + (pack + predict) + pack + L-BFGS-B init
        # + per round (K2 + stepper) + results + select_best; fused: fit + pack + predict + 1 + select
        "gpu_launches": int(K * 5 + agg["rounds"]) if agg["fused"] else int(K * 7 + 2 * agg["rounds"]),
        "clocks": clocks,
        "strong": strong,
    }
    if cfg4 is not None:
        line["cfg4"] = cfg4
    if world == 1 and not args.no_cpu_baseline:
        line["cpu_baseline"] = cpu_baseline(wl, X, z, perms, w0)
        line["lstm"] = lstm_measure()
    print(json.dumps(line), flush=True)


def write_outputs(out_dir, arrays, suffix=""):
    """--dump-outputs: one DIR/<name><suffix>.npy per array, float32 kept, everything else as float64 (the integer
    outputs are far below 2**53, so exactly).  cfg 3, the largest workload, writes 29 MB."""
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        a = a.cpu().numpy() if hasattr(a, "cpu") else np.asarray(a)
        np.save(os.path.join(out_dir, name + suffix + ".npy"), a if a.dtype == np.float32 else a.astype(np.float64))


def cpu_baseline(wl, X, z, perms, w0):
    """The oracle port timed on ONE host core (the reference is single-process and serial),
    bounded: the full fit + a sample of the starts."""
    S_cpu = 1024 if wl["dims"][0] < 20 else 768
    X0 = np.random.RandomState(1).uniform(size=(S_cpu, wl["dims"][0]))
    tf, ta, ev = reference_step(wl, X, z, perms, w0, X0, None, 1)
    scale = wl["starts"] / S_cpu
    full = tf + ta * scale
    return {"value": ev * scale / full, "unit": "evals/s", "cores": 1, "kind": "port",
            "sample": f"1 process: full fit ({wl['epochs']} epochs, {tf:.2f} s) + {S_cpu} of "
                      f"{wl['starts']} starts ({ta:.1f} s, {ev} evals), extrapolated linearly in "
                      "starts; NumPy restatement of Keras + installed SciPy L-BFGS-B (not TF)",
            "argmax_evals_per_sec": ev / ta, "adam_steps_per_sec":
                wl["epochs"] * (-(-wl["N"] // wl["batch"])) / tf,
            "host_cores_available": os.cpu_count()}


def lstm_measure(steps=3, with_cpu=True):
    """SURVEY.md section 8f row 4, measured: one proposal of the LSTM multi-fidelity plugin on a synthetic
    record -- 400 configurations of an 8-D space over 4 rungs (successive halving: every rung keeps a third),
    fit for 100 Adam steps (the plugin's num_steps_per_iter), then the 1,024-sample / 5-start argmax on the
    one-to-one view of rung 2 -- through the public API, host clock.  With `with_cpu` (the cpu_baseline leg)
    the oracle port (NumPy restatement + SciPy L-BFGS-B, one core) does the same proposal next to it."""
    import torch
    from scipy.optimize import Bounds
    from bore_b200 import ops
    from bore_b200.layers import BinaryCrossentropy
    from bore_b200.models import StackedRecurrentFactory
    D, U, L, T, N, B, mv = 8, 32, 2, 4, 400, 64, -1.0
    rs = np.random.RandomState(0)
    X = np.repeat(rs.uniform(size=(N, 1, D)), T, axis=1)
    Y = (rs.uniform(size=(N, T, 1)) < 1 / 3).astype(np.float64)
    alive = N
    for t in range(T):  # configurations beyond the survivors of rung t are padded
        X[alive:, t] = mv
        Y[alive:, t] = mv
        alive = max(alive // 3, 1)
    epochs = 100 // (-(-N // B))
    perms = np.stack([rs.permutation(N) for _ in range(epochs)])
    bounds = Bounds(np.zeros(D), np.ones(D))
    fac = StackedRecurrentFactory(D, 1, num_layers=L, num_units=U, layer_kws=dict(activation="elu"), seed=1)
    net = fac.build_many_to_many(mask_value=mv)
    net.compile(optimizer="adam", loss=BinaryCrossentropy(from_logits=True), metrics=["accuracy"])
    one = fac.build_one_to_one(3, transform=ops.sigmoid)
    w0 = net.get_weights()  # Keras-default initialisers drawn by the factory (glorot / orthogonal / forget bias 1)

    def gpu_step():
        net.set_weights(w0)
        net.set_optimizer_state([np.zeros_like(a) for a in w0], [np.zeros_like(a) for a in w0], 0)
        t0 = time.perf_counter()
        h = net.fit(X, Y, epochs=epochs, batch_size=B, permutations=perms, verbose=0).history["loss"]
        t1 = time.perf_counter()
        r = one.argmax(bounds, num_starts=5, num_samples=1024, print_fn=None, random_state=np.random.RandomState(2))
        torch.cuda.synchronize()
        return t1 - t0, time.perf_counter() - t1, h, r
    gpu_step()
    tfs, tas = [], []
    for _ in range(steps):
        a, b, hist, res = gpu_step()
        tfs.append(a); tas.append(b)
    # medians: the argmax is ~10 rounds of two small launches each, and one host hiccup (5 ms -> 100 ms) in one of
    # three steps used to triple the mean
    tf, ta = float(np.median(tfs)) * steps, float(np.median(tas)) * steps
    rec = {"workload": f"LSTM{U}x{L} (elu) on {N} sequences x {T} rungs of an {D}-D space, {epochs} epochs x "
                       f"{-(-N // B)} steps, argmax 1,024 samples -> 5 starts at rung 2",
           "fit_ms": 1e3 * tf / steps, "argmax_ms": 1e3 * ta / steps, "proposals_per_sec": steps / (tf + ta),
           "argmax_value": float(-res.fun),
           "bound": "latency (one CTA trains; <= 5 starts optimise)", "timing": "host clock, public API, median of the steps"}
    if with_cpu:
        rec.update(lstm_cpu_port(w0, X, Y, epochs, B, perms, mv, bounds, np.array(hist)))
    return rec


def lstm_cpu_port(w0, X, Y, epochs, B, perms, mv, bounds, gpu_hist):
    """cpu_baseline leg of the LSTM record: the same proposal by the oracle port on one host core."""
    from scipy.optimize import minimize
    from oracle import keras_lstm as kl
    D = X.shape[2]
    w = [a.copy() for a in w0]
    t0 = time.perf_counter()
    h_ref, _ = kl.fit(w, "elu", X, Y, epochs, B, perms, mv)
    c_fit = time.perf_counter() - t0
    t0 = time.perf_counter()
    Xi = np.random.RandomState(2).uniform(size=(1024, D))
    zi = kl.predict_one_to_one(w, "elu", Xi, 3)[:, 0]
    ind = np.argpartition(-zi, kth=4)[:5]

    def fn(x):
        f, g = kl.value_and_input_grad(w, "elu", x[None], 3, "sigmoid", True, np.float32)
        return float(f[0]), g[0].astype(np.float64)
    best = min(minimize(fn, x0=Xi[i], jac=True, method="L-BFGS-B", bounds=bounds,
                        options=dict(maxiter=1000, ftol=1e-9)).fun for i in ind)
    c_arg = time.perf_counter() - t0
    return {"loss_vs_oracle_max_abs": float(np.abs(gpu_hist - h_ref).max()), "oracle_argmax_value": float(-best),
            "cpu_port": {"fit_ms": 1e3 * c_fit, "argmax_ms": 1e3 * c_arg, "cores": 1,
                         "proposals_per_sec": 1.0 / (c_fit + c_arg), "kind": "port"}}


def cfg4_measure(rank, local_rank, world, steps, warm):
    """BASELINE.json configs[3]: 4,096 independent BO problems (seeds of 6-D Hartmann) trained
    and maximised concurrently, problems sharded over the ranks with no collective.  A step =
    one BO iteration of EVERY problem (fit 125 epochs on 500 observations + 1,024-sample
    screening + 5-start L-BFGS-B each, the plugin defaults), timed on the host clock around the
    public API (numpy in/out).  Returns the record on rank 0, None elsewhere."""
    import torch
    import torch.distributed as dist
    from bore_b200 import BatchedMaximizableSequential, Dense, problem_shard
    torch.cuda.set_device(local_rank)
    total, N, D, E, B, K, P = 4096, 500, 6, 125, 64, 5, 1024
    lo_p, hi_p = problem_shard(total, rank, world)
    M = hi_p - lo_p
    dims = [6, 32, 32, 1]
    rs = np.random.RandomState(100 + rank)
    X = rs.uniform(size=(M, N, D))
    y = np.stack([hartmann6(X[p]) for p in range(M)])
    z = np.stack([y[p] < np.quantile(y[p], 0.25) for p in range(M)])
    perms = np.stack([np.random.RandomState(7).permutation(N) for _ in range(E)])
    rs_draw = np.random.RandomState(500 + rank)
    layers = [Dense(32, activation="relu", input_dim=D), Dense(32, activation="relu"),
              Dense(1, activation="sigmoid")]
    model = BatchedMaximizableSequential(layers, n_problems=M, seed=rank, device=local_rank)
    model.compile(optimizer="adam", loss="binary_crossentropy")
    model.set_weights([glorot_init(dims, 1000 + lo_p + p) for p in range(M)])
    params = model._net.params_tensor()
    w0d = params.clone()
    phase = dict(fit=0.0, argmax=0.0)

    def step(record=False):
        params.copy_(w0d)                 # the same work every step: same init, fresh optimizer
        model._net.reset_optimizer()
        t0 = time.perf_counter()
        model.fit(X, z, batch_size=B, epochs=E, permutations=perms)
        if record:
            torch.cuda.synchronize()
        t1 = time.perf_counter()
        # (the 1,024 screening samples of every problem are drawn inside the call, from one RandomState, as M
        #  sequential reference argmax calls would: host work that overlaps the training kernels)
        res = model.argmax([(0.0, 1.0)] * D, num_starts=K, num_samples=P, random_state=rs_draw)
        t2 = time.perf_counter()
        if record:
            phase["fit"] += t1 - t0; phase["argmax"] += t2 - t1
        return model._last_stats["evals"], int(res.found.sum())

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
    sampler = ClockSampler(local_rank if rank == 0 else None)
    sampler.start()  # (before the warm-up, rank 0 only: see run_ours)
    for _ in range(warm):
        step()
    barrier()
    t0 = time.perf_counter()
    evals = 0
    for _ in range(steps):
        e, found = step()
        evals += e
    barrier()
    dt = time.perf_counter() - t0
    clocks = sampler.stop()
    step(record=True)                     # one extra step with a sync between the phases
    t = torch.tensor([dt, float(evals)], dtype=torch.float64, device="cuda")
    if world > 1:
        a = t.clone(); dist.all_reduce(a, op=dist.ReduceOp.MAX)
        b = t.clone(); dist.all_reduce(b, op=dist.ReduceOp.SUM)
        dt, evals = a[0].item(), b[1].item()
    if rank != 0:
        return None
    return {"metric": "bo_iterations_per_sec", "value": total * steps / dt, "unit": "BO iterations/s",
            "n_gpus": world, "steps": steps, "warmup": warm,
            "ms_per_step": 1e3 * dt / steps, "higher_is_better": True, "scaling": "strong",
            "vs_baseline": None, "dtype": "f32 MLP / f64 L-BFGS-B", "data": "synthetic",
            "config": {"workload": "4096 independent Hartmann-6 BO problems / Dense32x2-ReLU+sigmoid / "
                                   "N=500, 125 epochs, 1024 samples -> 5 starts each"},
            "notes": {"parallelism": f"problems sharded x{world}, no collective",
                      "timing": "host clock around the public API (numpy in/out), i.e. end to end",
                      "phases": "phases_ms_rank0 comes from ONE extra step with a synchronize between fit and argmax; "
                                "there the host-side draw of the 1,024 screening samples per problem no longer "
                                "overlaps the training kernels, so the two phases add up to more than ms_per_step"},
            "phases_ms_rank0": {"fit": 1e3 * phase["fit"], "argmax": 1e3 * phase["argmax"]},
            "evals_per_sec": evals / dt, "found_last_step": found, "clocks": clocks}


def run_cfg4(args, rank, local_rank, world):
    line = cfg4_measure(rank, local_rank, world, steps=args.steps, warm=max(1, min(args.warmup, 2)))
    if line is not None:
        print(json.dumps(line), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="cfg3", choices=sorted(WORKLOADS) + ["cfg4"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-cfg4", action="store_true", help="skip the short cfg 4 sub-record")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the last timed step computed to DIR/<name>.npy (inputs are seeded, so two "
                         "builds can be compared output for output)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "ours" or args.workload == "cfg4"):
        ap.error("--dump-outputs is for the GPU arm of cfg2 / cfg3 / cfg5")
    from bore_b200 import distributed as bd
    rank, local_rank, world = bd.env_world()
    if args.workload == "cfg4":
        if world > 1:
            bd.init_process_group("nccl")
        run_cfg4(args, rank, local_rank, world)
        if world > 1:
            import torch.distributed as dist
            dist.barrier()
            dist.destroy_process_group()
        return
    wl = WORKLOADS[args.workload]
    if args.impl == "reference":
        run_reference(args, wl, rank, world)
        return
    if world > 1:
        bd.init_process_group("nccl")
    run_ours(args, wl, rank, local_rank, world)
    if world > 1:
        import torch.distributed as dist
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
