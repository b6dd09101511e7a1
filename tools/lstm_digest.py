"""Bit-for-bit fingerprint of the LSTM kernels (csrc/lstm.cu) on the nets of tests/test_gpu_lstm.py.

For every net of that file's CASES (and one net with an extended activation, so that every build of
lstm_fit_kernel runs): a fit under Adam and one under Nadam with l1 + l2 penalties -- epoch losses,
trained weights, optimizer state --, the many-to-many logits with masking, and value + input gradient
of the one-to-one network under the three transforms.  Every array is written as .npy under OUT, and
one SHA-256 over all of them in name order to OUT/digest.txt.  Two trees whose kernels compute the same
thing print the same digest.

    python tools/lstm_digest.py OUT
"""
import hashlib
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "tests")]


def _sequences(rs, N, T, D, mv):
    X = rs.uniform(size=(N, T, D))
    Y = (rs.uniform(size=(N, T, 1)) < 0.4).astype(np.float64)
    for n in range(N):
        first = n % 3 == 0
        keep = rs.randint(first + 1, T + 1)
        X[n, :first] = mv; Y[n, :first] = mv
        X[n, keep:] = mv; Y[n, keep:] = mv
    X[5, 1] = mv; Y[5, 1] = mv  # a gap
    return X, Y


def run(out):
    from oracle import keras_lstm as kl
    from bore_b200 import layers, ops
    from bore_b200.models import StackedRecurrentFactory
    from test_gpu_lstm import CASES
    arrays = {}
    for D, U, L, act in list(CASES) + [(8, 32, 2, "selu")]:
        tag = f"{D}_{U}_{L}_{act}"
        for opt in ("adam", "nadam_l1"):
            reg = layers.l1_l2(1e-4, 1e-4) if opt == "nadam_l1" else None
            fac = StackedRecurrentFactory(D, 1, num_layers=L, num_units=U, seed=0,
                                          layer_kws=dict(activation=act, kernel_regularizer=reg,
                                                         bias_regularizer=reg))
            net = fac.build_many_to_many(mask_value=-1.0)
            net.compile(optimizer="adam" if opt == "adam" else layers.Nadam(),
                        loss=layers.BinaryCrossentropy(from_logits=True), metrics=["accuracy"])
            net.set_weights(kl.init_weights(D, U, L, seed=11))
            rs = np.random.RandomState(D * 100 + U)
            X, Y = _sequences(rs, 70, 4, D, -1.0)
            perms = np.stack([rs.permutation(70) for _ in range(6)])
            key = f"{tag}_{opt}"
            arrays[f"{key}_loss"] = np.asarray(
                net.fit(X, Y, epochs=6, batch_size=32, permutations=perms, verbose=0).history["loss"])
            for i, w in enumerate(net.get_weights()):
                arrays[f"{key}_w{i:02d}"] = w
            state = net.get_optimizer_state()
            for i, (m, v) in enumerate(zip(state[0], state[1])):
                arrays[f"{key}_m{i:02d}"] = m
                arrays[f"{key}_v{i:02d}"] = v
            arrays[f"{key}_iterations"] = np.asarray([state[2]] + list(state[3:]), np.float64)
            arrays[f"{key}_evaluate"] = np.asarray(net.evaluate(X, Y), np.float64)
            arrays[f"{key}_logits"] = net.predict(X)
            Xs = rs.uniform(size=(300, D))
            for T in (1, 4, 8):
                arrays[f"{key}_one_to_one_T{T}"] = fac.build_one_to_one(T).predict(Xs)
                for tr in ("identity", "sigmoid", "exp"):
                    f, g = fac.build_one_to_one(T, transform=ops.TRANSFORMS[tr])._func_min(Xs)
                    arrays[f"{key}_f_T{T}_{tr}"] = np.asarray(f)
                    arrays[f"{key}_g_T{T}_{tr}"] = np.asarray(g)
    os.makedirs(out, exist_ok=True)
    h = hashlib.sha256()
    for name in sorted(arrays):
        a = np.ascontiguousarray(arrays[name])
        np.save(os.path.join(out, name + ".npy"), a)
        h.update(name.encode()); h.update(str(a.dtype).encode()); h.update(str(a.shape).encode())
        h.update(a.tobytes())
    digest = h.hexdigest()
    with open(os.path.join(out, "digest.txt"), "w") as fh:
        fh.write(f"{digest}  {len(arrays)} arrays\n")
    print(digest, len(arrays), "arrays")


if __name__ == "__main__":
    run(sys.argv[1])
