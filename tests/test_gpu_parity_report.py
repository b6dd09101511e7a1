"""Parity report over BASELINE.json's five configurations, written as JSON to the file that
BORE_PARITY_REPORT names (nothing is written without it: a test run leaves the tree as it was;
profiles/parity_r02.json is one such report).  Per configuration:

  * fit: the CUDA training kernel against the NumPy oracle from the same initial weights and
    minibatch permutations -- max |loss difference| per epoch against the fp32 oracle and the
    fp64 oracle, next to the fp32-vs-fp64 difference of the ORACLE itself (the yardstick once
    rounding noise has been amplified through ReLU kinks);
  * argmax: >= 2,048 starts minimised on the device and by SciPy L-BFGS-B on the oracle MLP with
    the SAME (device-trained) weights: two-sided agreement (|dfun| <= 1e-4, north_star), one-sided
    agreement (ours <= reference + 1e-4), the reference's agreement with ITSELF under an fp32
    re-association of the MLP (hidden units permuted), and the status histograms.

The gates are what the numbers support (VERDICT r1, item 4): within 3 points of the reference's
self-agreement (or >= 0.95 ReLU / 0.99 ELU outright), ABNORMAL rates within 3 points.
"""
import json
import os
import multiprocessing as mp

import numpy as np
import pytest

from oracle import keras_mlp as km, argmax as am
from helpers import permuted_units, fork_pool

pytestmark = pytest.mark.gpu

FUN_TOL = 1e-4
S_STARTS = 2048


def _branin(X):
    x1 = -5.0 + 15.0 * X[:, 0]
    x2 = 15.0 * X[:, 1]
    b, c, r, s, t = 5.1 / (4 * np.pi ** 2), 5 / np.pi, 6.0, 10.0, 1 / (8 * np.pi)
    return (x2 - b * x1 ** 2 + c * x1 - r) ** 2 + s * (1 - t) * np.cos(x1) + s


_H_A = np.array([[10, 3, 17, 3.5, 1.7, 8], [0.05, 10, 17, 0.1, 8, 14], [3, 3.5, 1.7, 10, 17, 8],
                 [17, 8, 0.05, 10, 0.1, 14]])
_H_P = 1e-4 * np.array([[1312, 1696, 5569, 124, 8283, 5886], [2329, 4135, 8307, 3736, 1004, 9991],
                        [2348, 1451, 3522, 2883, 3047, 6650], [4047, 8828, 8732, 5743, 1091, 381]])


def _hartmann6(X):
    al = np.array([1.0, 1.2, 3.0, 3.2])
    inner = np.einsum("ij,nij->ni", _H_A, (X[:, None, :] - _H_P[None]) ** 2)
    return -np.sum(al * np.exp(-inner), axis=1)


def _ackley(X):
    u = -32.768 + 65.536 * X
    d = X.shape[1]
    return (-20.0 * np.exp(-0.2 * np.sqrt(np.sum(u * u, axis=1) / d))
            - np.exp(np.sum(np.cos(2 * np.pi * u), axis=1) / d) + 20.0 + np.e)


def _plugin8(X):
    return _ackley(X) + 0.3 * np.sin(7.0 * X[:, 0])


CONFIGS = {
    "cfg1": dict(dims=[2, 16, 16, 1], acts=["relu", "relu", "sigmoid"], transform="identity",
                 target=_branin, N=110, epochs=200, gamma=0.25, relu=True),
    "cfg2": dict(dims=[6, 32, 32, 1], acts=["relu", "relu", "sigmoid"], transform="identity",
                 target=_hartmann6, N=500, epochs=125, gamma=0.25, relu=True),
    "cfg3": dict(dims=[50, 64, 64, 64, 1], acts=["relu", "relu", "relu", "sigmoid"], transform="identity",
                 target=_ackley, N=2000, epochs=31, gamma=0.25, relu=True),
    # cfg 4 = cfg 2's network for independent problems: other seeds of the same problem
    "cfg4": dict(dims=[6, 32, 32, 1], acts=["relu", "relu", "sigmoid"], transform="identity",
                 target=_hartmann6, N=500, epochs=125, gamma=0.25, relu=True, seed=4242),
    "cfg5": dict(dims=[8, 32, 32, 32, 1], acts=["elu", "elu", "elu", "linear"], transform="sigmoid",
                 target=_plugin8, N=500, epochs=125, gamma=1 / 3, relu=False),
}


def _ref_chunk(args):
    w, acts, X0, transform = args
    from scipy.optimize import Bounds
    from threadpoolctl import threadpool_limits
    n = X0.shape[1]
    with threadpool_limits(1):
        return am.minimize_starts(w, acts, X0, Bounds(np.zeros(n), np.ones(n)), transform=transform)


def _reference(w, acts, X0, transform, pool, parts):
    outs = pool.map(_ref_chunk, [(w, acts, c, transform) for c in np.array_split(X0, parts) if len(c)])
    return {k: np.concatenate([o[k] for o in outs]) for k in ("fun", "status", "nit", "nfev")}


@pytest.fixture(scope="module")
def report():
    rep = {"fun_tol": FUN_TOL, "starts_per_config": S_STARTS,
           "oracle": "NumPy restatement of Keras (unpinned: no TensorFlow in the image) + the installed "
                     "SciPy L-BFGS-B (pinned)", "configs": {}}
    yield rep
    path = os.environ.get("BORE_PARITY_REPORT")
    if path:
        with open(path, "w") as f:
            f.write(json.dumps(rep, indent=1))


@pytest.mark.parametrize("name", sorted(CONFIGS))
def test_config_parity(name, report):
    from bore_b200.engine import NativeMLP
    c = CONFIGS[name]
    dims, acts, transform = c["dims"], c["acts"], c["transform"]
    n = dims[0]
    seed = c.get("seed", 0)
    rs = np.random.RandomState(seed)
    X = rs.uniform(size=(c["N"], n))
    y = c["target"](X)
    z = y < np.quantile(y, c["gamma"])
    E = c["epochs"]
    perms = np.stack([rs.permutation(c["N"]) for _ in range(E)]).astype(np.int32)
    w0 = km.init_weights(dims, seed)

    # ---- fit ----
    net = NativeMLP(dims, acts)
    net.set_weights(w0)
    hist = net.fit(X, z, E, 64, perms)
    w32 = [a.copy() for a in w0]
    h32, _ = km.fit(w32, acts, X, z, E, 64, perms)
    w64 = [a.astype(np.float64) for a in w0]
    h64, _ = km.fit(w64, acts, X, z, E, 64, perms, dtype=np.float64)
    d_gpu32 = np.abs(hist - h32)
    d_gpu64 = np.abs(hist.astype(np.float64) - h64)
    d_or = np.abs(h32.astype(np.float64) - h64)
    first_bad = int(np.argmax(d_gpu32 > 1e-4)) if (d_gpu32 > 1e-4).any() else E
    fit_rec = dict(epochs=E, adam_steps=E * (-(-c["N"] // 64)),
                   max_abs_dloss_vs_fp32_oracle=float(d_gpu32.max()),
                   max_abs_dloss_vs_fp64_oracle=float(d_gpu64.max()),
                   oracle_fp32_vs_fp64=float(d_or.max()),
                   epochs_within_1e4_of_fp32_oracle=first_bad,
                   per_epoch_vs_fp32_oracle=[float(v) for v in d_gpu32],
                   per_epoch_vs_fp64_oracle=[float(v) for v in d_gpu64],
                   per_epoch_oracle_fp32_vs_fp64=[float(v) for v in d_or])

    # ---- argmax on the device-trained weights ----
    w = net.get_weights()
    X0 = np.random.RandomState(seed + 1).uniform(size=(S_STARTS, n))
    got = net.lbfgsb(X0, 0.0, 1.0, transform=transform)
    cores = max(1, min(os.cpu_count() or 1, 32))
    with fork_pool(cores) as pool:
        ref = _reference(w, acts, X0, transform, pool, cores * 2)
        alt = _reference(permuted_units(w), acts, X0, transform, pool, cores * 2)
    agree = np.abs(got["fun"] - ref["fun"]) <= FUN_TOL
    one_sided = got["fun"] <= ref["fun"] + FUN_TOL
    r_self = np.abs(alt["fun"] - ref["fun"]) <= FUN_TOL
    r_self_one = alt["fun"] <= ref["fun"] + FUN_TOL
    arg_rec = dict(starts=S_STARTS, agree=float(agree.mean()), one_sided=float(one_sided.mean()),
                   reference_self_agreement=float(r_self.mean()),
                   reference_self_one_sided=float(r_self_one.mean()),
                   agree_within_1e3=float(np.mean(np.abs(got["fun"] - ref["fun"]) <= 1e-3)),
                   status_hist_ours=np.bincount(got["status"], minlength=3).tolist(),
                   status_hist_reference=np.bincount(ref["status"], minlength=3).tolist(),
                   status_hist_reference_reassociated=np.bincount(alt["status"], minlength=3).tolist(),
                   nit_mean=(float(got["nit"].mean()), float(ref["nit"].mean())),
                   nfev_mean=(float(got["nfev"].mean()), float(ref["nfev"].mean())),
                   mean_fun=(float(got["fun"].mean()), float(ref["fun"].mean())),
                   best_fun=(float(got["fun"].min()), float(ref["fun"].min())),
                   path="fused persistent kernel" if got["rounds"] == 1 else "lock-step rounds")
    report["configs"][name] = dict(network=f"{dims} {acts} transform={transform}", fit=fit_rec, argmax=arg_rec)
    print(name, {k: v for k, v in fit_rec.items() if not k.startswith("per_epoch")}, arg_rec)

    # ---- gates ----
    # fit: 1e-4 (north_star) wherever the oracle itself is reproducible; overall no further from the
    # fp64 oracle than twice what the fp32 oracle is (the rounding noise both share)
    assert d_gpu64.max() <= max(1e-4, 2.0 * d_or.max()) + 1e-6, (d_gpu64.max(), d_or.max())
    # the yardstick is the reference's agreement with ITSELF under an fp32 re-association: on ReLU
    # nets, and on saturated sigmoid-transformed ELU nets too (cfg 5 trained for 125 epochs: the
    # fp32 objective has plateaus; SciPy agrees with itself on 90 % of the starts only), an ulp
    # sends a start to another stationary point
    target = 0.95 if c["relu"] else 0.99
    assert agree.mean() >= min(target, r_self.mean() - 0.03), (agree.mean(), r_self.mean())
    assert one_sided.mean() >= min(0.93, r_self_one.mean() - 0.03), (one_sided.mean(), r_self_one.mean())
    # the ABNORMAL rate (results the reference's argmax drops, bore/mixins.py:85) must match too
    # -- up to 3 points plus the swing the reference's own rate shows under the re-association (cfg 1, two sets of
    # trained weights: reference 99 / 101 of 2,048 with the re-associated net, ours 145; reference 72 / 115, ours 166)
    ab_o, ab_r, ab_a = np.mean(got["status"] == 2), np.mean(ref["status"] == 2), np.mean(alt["status"] == 2)
    assert abs(ab_o - ab_r) <= 0.03 + abs(ab_a - ab_r), (ab_o, ab_r, ab_a)


def test_smooth_objective_sample_of_65536(report):
    """cfg 5 (plugin defaults, ELU) at 65,536 starts: a sample of 2,048 against SciPy, >= 0.99."""
    from bore_b200.engine import NativeMLP
    from helpers import trained_weights
    c = CONFIGS["cfg5"]
    dims, acts, transform = c["dims"], c["acts"], c["transform"]
    w = trained_weights(dims, acts, seed=5)
    net = NativeMLP(dims, acts)
    net.set_weights(w)
    S = 65536
    X0 = np.random.RandomState(5).uniform(size=(S, dims[0]))
    got = net.lbfgsb(X0, 0.0, 1.0, transform=transform)
    idx = np.random.RandomState(6).choice(S, S_STARTS, replace=False)
    cores = max(1, min(os.cpu_count() or 1, 32))
    with fork_pool(cores) as pool:
        ref = _reference(w, acts, X0[idx], transform, pool, cores * 2)
    agree = np.abs(got["fun"][idx] - ref["fun"]) <= FUN_TOL
    assert got["nit"].mean() >= 3.0  # a real optimisation, not a flat objective
    report["cfg5_65536_sample"] = dict(total_starts=S, sample=S_STARTS, agree=float(agree.mean()),
                                       nit_mean=float(got["nit"].mean()), nfev_mean=float(got["nfev"].mean()),
                                       max_abs_dfun=float(np.abs(got["fun"][idx] - ref["fun"]).max()),
                                       status_hist_ours=np.bincount(got["status"], minlength=3).tolist(),
                                       status_hist_reference_sample=np.bincount(ref["status"], minlength=3).tolist())
    print("cfg5 65536 sample", report["cfg5_65536_sample"])
    assert agree.mean() >= 0.99
